/*
 * plane_jobs.cpp -- the per-plane job descriptors of one picture and the lane buffers they point at, filled and
 * allocated the same way by the engines (encoder.cpp, decoder.cpp) and by the batch entry points of the kernel-level
 * API (kernel_api.cu) that check them.
 */
#include "engine.h"

namespace dsv {

void enc_fill_plane(SbtJob *s, HzJob *h, const CodecGeom &g, int p, int k, int isP, int quant, const EncPlaneIO &io)
{
    memset(s, 0, sizeof(*s));
    sbt_fill_geometry(s, g.pw[p], g.ph[p], g.cw[p], g.ch[p], isP, p);
    sbt_fill_quant(s, quant, isP, p, g.nbh, g.nbv);
    s->pix = const_cast<uint8_t *>(io.in);
    s->pstride = io.in_stride;
    s->opix = io.out;
    s->ostride = io.out_stride;
    if (isP) {
        s->addp = io.pred;
        s->addstride = io.pred_stride;
    }
    s->coef = io.coef;
    s->llx = io.llx;
    s->dv = io.dv;
    s->tflags = io.tflags ? io.tflags + (p > 0 ? g.tiles[0] : 0) + (p > 1 ? g.tiles[1] : 0) : nullptr;
    s->stable = io.stable;
    s->do_quant = 1;

    memset(h, 0, sizeof(*h));
    h->cw = g.cw[p];
    h->ch = g.ch[p];
    h->plane = p;
    h->isP = isP;
    h->pq = s->pq;
    h->dg = s->dg;
    hz_fill_regions(&h->rg, g.cw[p], g.ch[p]);
    h->nchunks = g.chunks[p];
    h->coef = s->coef;
    h->dv = s->dv;
    h->tflags = s->tflags;
    h->tiles_x = ceil_div(g.cw[p], SBT_TW);
    /* list scratch: the pack pass then reads no coefficient.  P pictures have a handful of dense chunks at most; those
     * are walked again rather than paying for the dense pack kernel's launch */
    h->dense = io.hz_dense ? io.hz_dense + (size_t) ((p > 0 ? g.chunks[0] : 0) + (p > 1 ? g.chunks[1] : 0)) * HZ_DENSE_BYTES : nullptr;
    h->list_mode = isP ? HZ_LISTS_SPARSE : HZ_LISTS_BOTH;
    h->stable = s->stable;
    h->chunk_base = k * g.total_chunks + (p > 0 ? g.chunks[0] : 0) + (p > 1 ? g.chunks[1] : 0);
    h->frame = k;
}

size_t enc_packet_cap(const CodecGeom &g)
{
    /* The reference sizes its packet by a heuristic (w*h*{2,4,6}, dsv_encoder.c:472-491) that noise-like content at
     * top quality can exceed.  Here the bound is structural: a coefficient costs at most UEG(run = 0) + NEG(symbol)
     * = 1 + 2 * 17 + 2 bits for symbols below 2^17 (8-bit samples through 6 levels of 3.2x LL gain, divided by a
     * quantiser >= 16, stay below 2^14), i.e. < 4.75 bytes; hzcc_prefix_kernel refuses what still would not fit. */
    size_t ub = (size_t) g.w * g.h;
    ub *= (g.subsamp == DSV_SUBSAMP_444) ? 6 : (g.subsamp == DSV_SUBSAMP_422) ? 4 : 2;
    const size_t cap = ub + 4096 + (size_t) g.nblk * 48;
    const size_t bound = g.coef_total * 19 / 4 + 4096 + (size_t) g.nblk * 48;
    return ((cap > bound ? cap : bound) + 255) & ~(size_t) 255;
}

void enc_fill_frame(HzFrame *f, uint8_t *pkt, unsigned cap, unsigned start_byte, int k)
{
    memset(f, 0, sizeof(*f));
    f->pkt = pkt;
    f->cap = cap;
    f->start_byte = start_byte;
    f->nplanes = 3;
    f->job[0] = 3 * k;
    f->job[1] = 3 * k + 1;
    f->job[2] = 3 * k + 2;
}

void sse_fill_picture(SseJob *j, const CodecGeom &g, const DevFrame &src, const DevFrame &rec, unsigned long long *out)
{
    for (int p = 0; p < 3; p++) {
        j[p].src = src.p[p];
        j[p].src_stride = src.stride[p];
        j[p].rec = rec.p[p];
        j[p].rec_stride = rec.stride[p];
        j[p].pw = g.pw[p];
        j[p].ph = g.ph[p];
        j[p].out = out + p;
    }
}

int64_t ssim_windows(int pw, int ph)
{
    return pw >= 8 && ph >= 8 ? (int64_t) (pw / 4 - 1) * (ph / 4 - 1) : 0;
}

void dec_fill_plane(SbtJob *s, HzJob *h, HzCleanItem *c, const CodecGeom &g, int p, int isP, int quant, const DevFrame &cur,
                    int32_t *coef, int32_t *llx, uint8_t *tflags, const uint8_t *stable)
{
    memset(s, 0, sizeof(*s));
    sbt_fill_geometry(s, g.pw[p], g.ph[p], g.cw[p], g.ch[p], isP, p);
    sbt_fill_quant(s, quant, isP, p, g.nbh, g.nbv);
    s->pix = s->opix = cur.p[p];
    s->pstride = s->ostride = cur.stride[p];
    s->coef = coef + g.coef_off[p];
    s->llx = llx;
    s->stable = stable;
    s->tflags = tflags + (p > 0 ? g.tiles[0] : 0) + (p > 1 ? g.tiles[1] : 0);
    memset(h, 0, sizeof(*h));
    h->cw = g.cw[p];
    h->ch = g.ch[p];
    h->plane = p;
    h->isP = isP;
    h->pq = s->pq;
    h->dg = s->dg;
    hz_fill_regions(&h->rg, g.cw[p], g.ch[p]);
    h->coef = s->coef;
    h->stable = s->stable;
    h->tflags = s->tflags;
    h->tiles_x = s->tiles_x;
    /* dsv_decoder.c:405: coefficient planes start zeroed.  Planes that were never coded (corrupt plen) stay all-zero
     * here; the reference leaves the zeroed residual plane untouched instead. */
    hzdec_fill_clean(c, *h, s->tiles_y);
}

void dec_init_flags(uint8_t *d_tflags, const CodecGeom &g)
{
    for (int p = 0, off = 0; p < 3; off += g.tiles[p], p++) {
        SbtJob probe;
        memset(&probe, 0, sizeof(probe));
        sbt_fill_geometry(&probe, g.pw[p], g.ph[p], g.cw[p], g.ch[p], 1, p);
        CUDA_CHECK(cudaMemset(d_tflags + off, hz_flag_base(probe.dg), (size_t) g.tiles[p] + (p == 2 ? 16 : 0)));
    }
}

void enc_lane_alloc(EncLane &l, const CodecGeom &g, bool inter, int levels, size_t pkt_bytes)
{
    CUDA_CHECK(cudaMalloc(&l.coef, g.coef_total * sizeof(int32_t)));
    CUDA_CHECK(cudaMalloc(&l.tflags, (size_t) g.total_tiles + 16));
    CUDA_CHECK(cudaMemset(l.tflags, 3, (size_t) g.total_tiles + 16));
    CUDA_CHECK(cudaMalloc(&l.hz_dense, (size_t) g.total_chunks * HZ_DENSE_BYTES));
    for (int p = 0; p < 3; p++) {
        CUDA_CHECK(cudaMalloc(&l.llx[p], sbt_llx_elems(g.cw[p], g.ch[p]) * sizeof(int32_t)));
        CUDA_CHECK(cudaMalloc(&l.dv[p], sbt_dv_elems(g.cw[p], g.ch[p]) * sizeof(int32_t)));
        CUDA_CHECK(cudaMemset(l.dv[p], 0, sbt_dv_elems(g.cw[p], g.ch[p]) * sizeof(int32_t)));
    }
    l.pkt_cap = pkt_bytes;
    CUDA_CHECK(cudaMalloc(&l.d_pkt, pkt_bytes));
    CUDA_CHECK(cudaMemset(l.d_pkt, 0, pkt_bytes));
    CUDA_CHECK(cudaMallocHost(&l.h_head, head_capacity(g)));
    devframe_alloc(&l.xf, g.w, g.h, g.subsamp);
    if (inter) {
        devframe_alloc(&l.pred, g.w, g.h, g.subsamp);
        for (int i = 0; i < 2; i++) {
            devframe_alloc(&l.pad[i], g.w, g.h, g.subsamp);
            devframe_alloc(&l.recon[i], g.w, g.h, g.subsamp);
            for (int k = 0; k < levels; k++) {
                devframe_alloc(&l.pyr[i][k], ceil_shift(g.w, k + 1), ceil_shift(g.h, k + 1), g.subsamp);
            }
        }
        for (int k = 1; k <= levels; k++) {
            CUDA_CHECK(cudaMalloc(&l.d_mvf[k], sizeof(DevMV) * (size_t) g.nblk));
            CUDA_CHECK(cudaMemset(l.d_mvf[k], 0, sizeof(DevMV) * (size_t) g.nblk));
        }
        CUDA_CHECK(cudaMalloc(&l.d_aux, sizeof(int2) * (size_t) g.nblk));
    }
}

void enc_lane_free(EncLane &l)
{
    cudaFree(l.coef);
    cudaFree(l.tflags);
    cudaFree(l.hz_dense);
    for (int p = 0; p < 3; p++) {
        cudaFree(l.llx[p]);
        cudaFree(l.dv[p]);
    }
    cudaFree(l.d_pkt);
    cudaFreeHost(l.h_head);
    devframe_free(&l.xf);
    devframe_free(&l.pred);
    devframe_free(&l.qrec);
    for (int i = 0; i < 2; i++) {
        devframe_free(&l.pad[i]);
        devframe_free(&l.recon[i]);
        for (int k = 0; k < DSV_MAX_PYRAMID_LEVELS; k++) {
            devframe_free(&l.pyr[i][k]);
        }
    }
    for (int k = 1; k <= DSV_MAX_PYRAMID_LEVELS; k++) {
        cudaFree(l.d_mvf[k]);
    }
    cudaFree(l.d_aux);
}

void dec_lane_alloc(DecLane &l, const CodecGeom &g)
{
    /* coefficient planes are kept all-zero between pictures by the flag-guided clean-up (hzdec_clean_kernel) */
    CUDA_CHECK(cudaMalloc(&l.coef, g.coef_total * sizeof(int32_t)));
    CUDA_CHECK(cudaMemset(l.coef, 0, g.coef_total * sizeof(int32_t)));
    CUDA_CHECK(cudaMalloc(&l.tflags, (size_t) g.total_tiles + 16));
    dec_init_flags(l.tflags, g);
    for (int p = 0; p < 3; p++) {
        CUDA_CHECK(cudaMalloc(&l.llx[p], sbt_llx_elems(g.cw[p], g.ch[p]) * sizeof(int32_t)));
        HzDecPlan pl;
        hzdec_plan(&pl, g.cw[p], g.ch[p]);
        hzdec_plane_alloc(&l.hz[p], pl);
    }
    devframe_alloc(&l.out[0], g.w, g.h, g.subsamp);
    devframe_alloc(&l.out[1], g.w, g.h, g.subsamp);
    /* packets are staged lazily: most are far smaller than the format's upper bound */
}

void dec_lane_free(DecLane &l)
{
    cudaFree(l.coef);
    cudaFree(l.tflags);
    for (int p = 0; p < 3; p++) {
        cudaFree(l.llx[p]);
        hzdec_plane_free(&l.hz[p]);
    }
    devframe_free(&l.out[0]);
    devframe_free(&l.out[1]);
    cudaFree(l.d_pkt);
    cudaFreeHost(l.h_pkt[0]);
    cudaFreeHost(l.h_pkt[1]);
    cudaFree(l.d_draw);
}

void ingest_fill_picture(IngestItem *it, const uint8_t *const src[3], const DevFrame &dst)
{
    for (int p = 0; p < 3; p++) {
        it[p].src = src[p];
        it[p].dst = plane_ref(dst, p);
    }
}

void down2_fill_level(Down2Item *it, const DevFrame &top, const DevFrame *pyr, int lv)
{
    it->src = plane_ref(lv == 0 ? top : pyr[lv - 1], 0);
    it->dst = plane_ref(pyr[lv], 0);
}

void sum_fill_lane(SumItem *it, const DevFrame *pyr, int levels, LaneMisc *d_misc, int lane)
{
    it->src = plane_ref(pyr[levels - 1], 0);
    it->out = &d_misc[lane].luma_sum;
}

void hme_fill_lane(HmeArgs *rows, int n_search, int q, const MotionGeom &mg, const DevFrame &src, const DevFrame *src_pyr,
                   const DevFrame &ref, const DevFrame *ref_pyr, DevMV *const *mvf, int2 *aux, LaneMisc *d_misc, int lane)
{
    DevFrame sf[DSV_MAX_PYRAMID_LEVELS + 1], rf[DSV_MAX_PYRAMID_LEVELS + 1];
    sf[0] = src;
    rf[0] = ref;
    for (int lv = 0; lv < mg.levels; lv++) {
        sf[lv + 1] = src_pyr[lv];
        rf[lv + 1] = ref_pyr[lv];
    }
    for (int lv = 0; lv <= mg.levels; lv++) {
        hme_fill_args(&rows[(size_t) lv * n_search + q], mg, lv, sf, rf, mvf, aux, &d_misc[lane].nintra);
    }
}

void enc_bmc_fill(BmcArgs *a, const MotionGeom &mg, const DevMV *mv, const DevFrame &recon_ref, const DevFrame &pred,
                  const DevFrame &src, const DevFrame &resid)
{
    bmc_fill_args(a, mg, mv, recon_ref, &pred, src, resid, 1);
}

void dec_bmc_fill(BmcArgs *list, int *n_p, int isP, const MotionGeom &mg, const DevMV *d_mv, int li, int nblk, const DevFrame &ref,
                  const DevFrame &cur)
{
    if (isP) {
        bmc_fill_args(&list[(*n_p)++], mg, d_mv + (size_t) li * nblk, ref, nullptr, cur, cur, 2);
    }
}

} // namespace dsv
