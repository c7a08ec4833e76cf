/*
 * decoder.cpp -- the dsv_decoder.h API (dsv_decoder.c:22-145,244-472) and the lock-step decode engine.
 *
 * Host code parses only what is serial and tiny: packet header, metadata, the ZBRLE stability map and
 * the four motion sub-streams (<= 2040 blocks), plus SEG(DC) / nruns / first run of each plane head.
 * Each lane's packet is copied to the device once; coefficient parsing (parallel bit-FSM), dequantisation,
 * the inverse subband transform, motion compensation + reconstruction and the border extension of the
 * new references run as kernels batched over all lanes, on the engine's stream:
 *   H2D packets -> zero coefs -> hzcc parse -> SBT inverse -> BMC + add (P) -> extend (refs) -> D2H pictures.
 * There is no CPU implementation of those stages in this library.
 */
#include "dsv1_b200.h"

#include "bits.h"
#include "engine.h"

using namespace dsv;

static int read_packet_hdr(BitReader &br) /* dsv_decoder.c:21-48 */
{
    int c0 = (int) br.get_bits(8), c1 = (int) br.get_bits(8), c2 = (int) br.get_bits(8), c3 = (int) br.get_bits(8);
    if (c0 != DSV_FOURCC_0 || c1 != DSV_FOURCC_1 || c2 != DSV_FOURCC_2 || c3 != DSV_FOURCC_3) {
        DSV_ERROR(("bad 4cc (%c %c %c %c)\n", c0, c1, c2, c3));
        return -1;
    }
    br.get_bits(8); /* minor version */
    int type = (int) br.get_bits(8);
    br.get_bits(32);
    br.get_bits(32);
    return type;
}

/* B.2.3.1 stability map (dsv_decoder.c:126-145) */
static void read_stability(BitReader &br, const uint8_t *pkt, unsigned pkt_len, uint8_t *stab, int nblk)
{
    br.align();
    unsigned len = br.get_ueg();
    br.align();
    unsigned at = br.byte_pos();
    RleReader rle(pkt + (at < pkt_len ? at : pkt_len), at < pkt_len ? pkt_len - at : 0);
    br.skip_bytes(len);
    for (int i = 0; i < nblk; i++) {
        stab[i] = (uint8_t) rle.get();
    }
}

/* B.2.3.2 motion data (dsv_decoder.c:72-124) */
static void read_motion(BitReader &br, const uint8_t *pkt, unsigned pkt_len, DevMV *mvs, uint8_t *stab, int nbh, int nbv)
{
    unsigned start[4];
    br.align();
    for (int s = 0; s < 4; s++) {
        unsigned len = br.get_ueg();
        br.align();
        start[s] = br.byte_pos() < pkt_len ? br.byte_pos() : pkt_len;
        br.skip_bytes(len);
    }
    RleReader mode(pkt + start[0], pkt_len - start[0]);
    BitReader bx(pkt + start[1], pkt_len - start[1]), by(pkt + start[2], pkt_len - start[2]);
    BitReader bm(pkt + start[3], pkt_len - start[3]);
    memset(mvs, 0, sizeof(DevMV) * (size_t) nbh * nbv);
    for (int j = 0; j < nbv; j++) {
        for (int i = 0; i < nbh; i++) {
            DevMV &mv = mvs[j * nbh + i];
            mv.mode = (uint8_t) mode.get();
            if (mv.mode == DSV_MODE_INTER) {
                int px, py;
                predict_mv(mvs, nbh, i, j, &px, &py);
                mv.x = (int16_t) (bx.get_seg() + px);
                mv.y = (int16_t) (by.get_seg() + py);
            } else {
                mv.submask = bm.get_bit() ? DSV_MASK_ALL_INTRA : (uint8_t) bm.get_bits(4);
                stab[j * nbh + i] |= 2;
            }
        }
    }
}

namespace dsv {

static bool host_packed(const CodecGeom &g, const OutRef &r)
{
    return !r.on_device && r.plane[0] && r.stride[0] == g.pw[0] && r.stride[1] == g.pw[1] && r.stride[2] == g.pw[2] &&
           r.plane[1] == r.plane[0] + g.plane_off[1] && r.plane[2] == r.plane[0] + g.plane_off[2];
}

/* dsv_decoder.c:383-413 */
int parse_plane_dir(const uint8_t *pkt, unsigned len, unsigned at, const CodecGeom &g, const uint8_t *d_pkt, HzPlaneData pd[3])
{
    BitReader br(pkt, len);
    br.skip_bytes(at);
    int n = 0;
    for (; n < 3; n++) {
        const int plen = (int) br.get_bits(32);
        const int framesz = g.cw[n] * g.ch[n] * (int) sizeof(int32_t);
        if (plen <= 0 || plen > framesz * 2) {
            DSV_ERROR(("plane length was strange: %d", plen));
            break;
        }
        const unsigned start = br.byte_pos();
        if (start >= len) {
            DSV_ERROR(("plane starts past the end of the packet"));
            break;
        }
        hzdec_parse_head(pkt + start, len - start, (unsigned) plen, &pd[n]);
        pd[n].body = d_pkt + start;
        br.skip_bytes((unsigned) plen);
    }
    return n;
}

DecEngine::DecEngine(const DSV_META &md, int lanes)
{
    CUDA_CHECK(cudaGetDevice(&device));
    plan_geometry(&g_, md.width, md.height, md.subsamp);
    plan_blocks(&g_, DSV_MIN_BLOCK_SIZE, DSV_MIN_BLOCK_SIZE); /* worst case; the real size is per picture */
    const CodecGeom &g = g_;
    max_nblk_ = g.nblk;
    L_ = lanes;
    if (const char *e = getenv("DSV_KERNEL_TIMES")) {
        time_kernels = atoi(e) != 0;
    }
    CUDA_CHECK(cudaStreamCreateWithFlags(&st_, cudaStreamNonBlocking));
    CUDA_CHECK(cudaStreamCreateWithFlags(&st_copy_, cudaStreamNonBlocking));
    for (int q = 0; q < 2; q++) {
        for (auto &e : ev_[q]) {
            CUDA_CHECK(cudaEventCreate(&e));
        }
        CUDA_CHECK(cudaEventCreateWithFlags(&ev_end_[q], cudaEventDisableTiming));
    }
    CUDA_CHECK(cudaEventCreateWithFlags(&ev_done_, cudaEventDisableTiming));
    CUDA_CHECK(cudaEventCreateWithFlags(&ev_copied_[0], cudaEventDisableTiming));
    CUDA_CHECK(cudaEventCreateWithFlags(&ev_copied_[1], cudaEventDisableTiming));
    /* a picture packet holds three planes of at most 2 * 4 * cw * ch bytes each (dsv_decoder.c:397-401) */
    pkt_cap_ = g.coef_total * 8 + 4096 + (size_t) g.nblk * 64;
    const size_t per_lane = 3 * (sizeof(SbtJob) + hzdec_job_size()) + sizeof(BmcArgs) + 8 * sizeof(PlaneRef) + 3 * sizeof(PackItem) + 3 * sizeof(HzCleanItem) + sizeof(CopyItem) + sizeof(DrawItem) + sizeof(PackItem) + 2 * sizeof(To420Item) + 1024;
    CUDA_CHECK(cudaMalloc(&d_mv_, sizeof(DevMV) * (size_t) max_nblk_ * L_));
    CUDA_CHECK(cudaMalloc(&d_stab_, (size_t) max_nblk_ * L_));
    for (int q = 0; q < 2; q++) {
        arena_[q].create(per_lane * (size_t) L_ + 4096);
        CUDA_CHECK(cudaMallocHost(&h_mv_[q], sizeof(DevMV) * (size_t) max_nblk_ * L_));
        CUDA_CHECK(cudaMallocHost(&h_stab_[q], (size_t) max_nblk_ * L_));
    }
    og_ = g_;
    {
        CodecGeom g420;
        plan_geometry(&g420, md.width, md.height, DSV_SUBSAMP_420);
        const size_t fb = g.frame_bytes > g420.frame_bytes ? g.frame_bytes : g420.frame_bytes;
        out_pitch_ = (fb + 255) & ~(size_t) 255;
    }
    CUDA_CHECK(cudaMalloc(&d_out_all_[0], out_pitch_ * L_ + 256));
    CUDA_CHECK(cudaMalloc(&d_out_all_[1], out_pitch_ * L_ + 256));
    lanes_.resize((size_t) L_);
    for (auto &l : lanes_) {
        dec_lane_alloc(l, g);
    }
}

DecEngine::~DecEngine()
{
    cudaStreamSynchronize(st_);
    cudaStreamSynchronize(st_copy_);
    for (auto &l : lanes_) {
        dec_lane_free(l);
    }
    arena_[0].destroy();
    arena_[1].destroy();
    cudaFree(d_out_all_[0]);
    cudaFree(d_out_all_[1]);
    cudaFree(d_mv_);
    cudaFreeHost(h_mv_[0]);
    cudaFreeHost(h_mv_[1]);
    cudaFree(d_stab_);
    cudaFreeHost(h_stab_[0]);
    cudaFreeHost(h_stab_[1]);
    for (int q = 0; q < 2; q++) {
        for (auto &e : ev_[q]) {
            cudaEventDestroy(e);
        }
        cudaEventDestroy(ev_end_[q]);
    }
    ktimes.destroy();
    cudaEventDestroy(ev_done_);
    cudaEventDestroy(ev_copied_[0]);
    cudaEventDestroy(ev_copied_[1]);
    cudaStreamDestroy(st_copy_);
    cudaStreamDestroy(st_);
}

void DecEngine::flush()
{
    CUDA_CHECK(cudaStreamSynchronize(st_));
    CUDA_CHECK(cudaStreamSynchronize(st_copy_));
    collect(0);
    collect(1);
}

/* the step that last used this parity's host buffers must have left the GPU before they are rewritten; its kernel
 * timings are read at the same moment */
void DecEngine::collect(int parity)
{
    Pending &pd = pending_[parity];
    if (!pd.valid) {
        return;
    }
    CUDA_CHECK(cudaEventSynchronize(ev_end_[parity]));
    ktimes.collect(parity);
    if (pd.timed) {
        float ms = 0;
        CUDA_CHECK(cudaEventElapsedTime(&ms, ev_[parity][0], ev_[parity][1]));
        stats.sbt_inv_ms += ms;
        stats.sbt_inv_launches++;
        unsigned long long bytes = 0;
        for (int p = 0; p < 3; p++) {
            bytes += (unsigned long long) g_.pw[p] * g_.ph[p] + 4ull * g_.cw[p] * g_.ch[p];
        }
        stats.sbt_inv_bytes += bytes * (unsigned) pd.pictures;
        if (pd.p_pictures) {
            CUDA_CHECK(cudaEventElapsedTime(&ms, ev_[parity][2], ev_[parity][3]));
            stats.bmc_ms += ms;
            stats.bmc_launches++;
            stats.bmc_bytes += 3ull * g_.frame_bytes * (unsigned) pd.p_pictures;
        }
    }
    stats.pictures += (unsigned) pd.pictures;
    pd.valid = false;
}

void DecEngine::set_out420(bool on)
{
    if (on && g_.subsamp != DSV_SUBSAMP_420) {
        plan_geometry(&og_, g_.w, g_.h, DSV_SUBSAMP_420);
    } else {
        og_ = g_;
    }
}

void DecEngine::step(int n, const int *lane_ids, const PktRef *pkts, const OutRef *out, int *codes, DSV_FNUM *fnums)
{
    cudaStream_t st = st_;
    const int par = (int) (step_no_ & 1);
    collect(par);
    const bool timed = time_kernels;
    KtActivate kt_on(timed ? &ktimes : nullptr);
    ktimes.open(par);
    StepArena &arena_ = this->arena_[par];
    uint8_t *const h_stab_ = this->h_stab_[par];
    DevMV *const h_mv_ = this->h_mv_[par];
    cudaEvent_t *const ev_ = this->ev_[par];
    int step_nblk = 0; /* lanes of a step share the block grid: vectors / stability bits are packed at that pitch */
    CodecGeom step_g = g_; /* that grid, planned from the step's first picture */
    arena_.reset();
    SbtJob *d_sj;
    void *d_hzj;
    BmcArgs *d_bmc;
    PlaneRef *d_ext;
    PackItem *d_pack;
    SbtJob *sj = arena_.push_n<SbtJob>((size_t) 3 * n, &d_sj);
    uint8_t *hzj = reinterpret_cast<uint8_t *>(arena_.push(hzdec_job_size() * (size_t) 3 * n, &d_hzj));
    BmcArgs *ba = arena_.push_n<BmcArgs>((size_t) n, &d_bmc);
    PlaneRef *ext = arena_.push_n<PlaneRef>((size_t) 3 * n, &d_ext);
    PackItem *pack = arena_.push_n<PackItem>((size_t) 3 * n, &d_pack);
    DrawItem *d_draw;
    DrawItem *draw = arena_.push_n<DrawItem>((size_t) n, &d_draw);
    PackItem *d_pack2;
    PackItem *pack2 = arena_.push_n<PackItem>((size_t) n, &d_pack2);
    To420Item *d_cv;
    To420Item *cv = arena_.push_n<To420Item>((size_t) 2 * n, &d_cv);
    int n_draw = 0, n_pack2 = 0, n_cv = 0;
    HzCleanItem *d_clean;
    HzCleanItem *clean = arena_.push_n<HzCleanItem>((size_t) 3 * n, &d_clean);
    int n_clean = 0;
    CopyItem *d_cpy;
    CopyItem *cpy = arena_.push_n<CopyItem>((size_t) n, &d_cpy);
    int n_cpy = 0;
    size_t max_cpy = 0;
    const double t_host0 = host_now_ms();
    HzDecDims dims;
    int n_sj = 0, n_p = 0, n_ext = 0, n_pack = 0;

    for (int k = 0; k < n; k++) {
        const int li = lane_ids[k];
        DecLane &l = lanes_[(size_t) li];
        const uint8_t *pkt = pkts[k].data;
        const unsigned pkt_len = pkts[k].len;
        codes[k] = DSV_DEC_ERROR;
        fnums[k] = (DSV_FNUM) -1;
        l.ok = 0;
        l.drawn = 0;
        BitReader br(pkt, pkt_len);
        const int pkt_type = read_packet_hdr(br);
        if (pkt_type == -1 || !DSV_PT_IS_PIC(pkt_type) || (size_t) pkt_len > pkt_cap_) {
            continue;
        }
        l.has_ref = DSV_PT_HAS_REF(pkt_type);
        l.is_ref = DSV_PT_IS_REF(pkt_type);
        br.align();
        l.fnum = br.get_bits(32);
        br.align();
        const int bw_ = (int) (br.get_ueg() << 2), bh_ = (int) (br.get_ueg() << 2);
        if (bw_ < DSV_MIN_BLOCK_SIZE || bh_ < DSV_MIN_BLOCK_SIZE || bw_ > DSV_MAX_BLOCK_SIZE || bh_ > DSV_MAX_BLOCK_SIZE) {
            continue;
        }
        CodecGeom g = g_;
        plan_blocks(&g, bw_, bh_);
        if (step_nblk == 0) {
            step_g = g;
        } else if (step_g.blk_w != bw_ || step_g.blk_h != bh_) {
            /* lanes of one step share the block grid (same format => same encoder choice); a stream that
             * deviates is decoded in a later step by its caller */
            DSV_ERROR(("mixed block sizes inside one batch step"));
            continue;
        }
        step_nblk = g.nblk;
        uint8_t *stab = h_stab_ + (size_t) li * step_nblk;
        DevMV *mvs = h_mv_ + (size_t) li * step_nblk;
        read_stability(br, pkt, pkt_len, stab, g.nblk);
        if (l.has_ref) {
            read_motion(br, pkt, pkt_len, mvs, stab, g.nbh, g.nbv);
        }
        br.align();
        l.quant = (int) br.get_bits(DSV_MAX_QP_BITS);

        /* packet bytes on the device */
        const uint8_t *d_pkt;
        if (pkts[k].dev_data) {
            d_pkt = pkts[k].dev_data;
        } else {
            if ((size_t) pkt_len + 80 > l.pkt_alloc) {
                /* staging grows with the largest packet seen (the format's upper bound, 8 bytes per coefficient,
                 * would pin hundreds of MB per lane at UHD); the previous step has completed, nothing is in flight */
                CUDA_CHECK(cudaStreamSynchronize(st)); /* earlier steps may still read the old staging */
                cudaFree(l.d_pkt);
                cudaFreeHost(l.h_pkt[0]);
                cudaFreeHost(l.h_pkt[1]);
                l.pkt_alloc = (size_t) pkt_len * 2 + (256 << 10);
                if (l.pkt_alloc > pkt_cap_ + 80) {
                    l.pkt_alloc = pkt_cap_ + 80;
                }
                CUDA_CHECK(cudaMalloc(&l.d_pkt, l.pkt_alloc));
                CUDA_CHECK(cudaMallocHost(&l.h_pkt[0], l.pkt_alloc));
                CUDA_CHECK(cudaMallocHost(&l.h_pkt[1], l.pkt_alloc));
            }
            uint8_t *h_pkt = l.h_pkt[par];
            memcpy(h_pkt, pkt, pkt_len);
            memset(h_pkt + pkt_len, 0, 64);
            cpy[n_cpy].dst = l.d_pkt;
            cpy[n_cpy].src = h_pkt;
            cpy[n_cpy].bytes = ((size_t) pkt_len + 64 + 15) & ~(size_t) 15;
            max_cpy = max_cpy > cpy[n_cpy].bytes ? max_cpy : cpy[n_cpy].bytes;
            n_cpy++;
            stats.h2d_bytes += pkt_len;
            d_pkt = l.d_pkt;
        }
        br.align();
        /* corrupt side-info lengths can carry the reader past the end, further than a 32-bit byte offset reaches */
        l.nplanes = parse_plane_dir(pkt, pkt_len, br.exhausted() ? pkt_len : br.byte_pos(), g, d_pkt, l.pd);
        fnums[k] = l.fnum;
        if (l.has_ref && !l.have_ref) {
            DSV_WARNING(("reference frame not found"));
            continue; /* DSV_DEC_ERROR (dsv_decoder.c:424-427) */
        }
        l.ok = 1;
        codes[k] = DSV_DEC_OK;

        const DevFrame &cur = l.out[l.cur];
        const int isP = l.has_ref;
        for (int p = 0; p < 3; p++) {
            HzJob h;
            dec_fill_plane(&sj[n_sj], &h, &clean[n_clean++], g, p, isP, l.quant, cur, l.coef, l.llx[p], l.tflags,
                           d_stab_ + (size_t) li * step_nblk);
            if (p < l.nplanes) {
                hzdec_fill_job(hzj + hzdec_job_size() * (size_t) dims.njobs, h, l.pd[p], l.hz[p], &dims);
            }
            n_sj++;
            if (l.is_ref) {
                ext[n_ext++] = plane_ref(cur, p);
            }
        }
        /*
         * Where the picture goes.  F[p]: dense destination in the OUTPUT format (the caller's device planes, or the
         * staging buffer a packed host destination is served from); strided destinations are copied straight from
         * the bordered frame later.  The overlay is painted on a dense copy, never on the frame the next picture
         * predicts from; -out420p converts chroma on the way out.
         */
        const CodecGeom &og = og_;
        const bool conv = og.subsamp != g.subsamp;
        const bool hostp = host_packed(og, out[k]);
        bool dense_out = true;
        for (int p = 0; p < 3; p++) {
            dense_out = dense_out && out[k].plane[p] && out[k].on_device && out[k].stride[p] == og.pw[p];
        }
        bool want_out = out[k].plane[0] != nullptr;
        if (conv && want_out && !dense_out && !hostp) {
            DSV_ERROR(("4:2:0 output needs a dense destination"));
            want_out = false;
        }
        l.noout = !want_out;
        l.drawn = draw_mode && isP && want_out;
        const bool scratch = l.drawn && (conv || (!dense_out && !hostp));
        if (scratch && !l.d_draw) {
            CUDA_CHECK(cudaMalloc(&l.d_draw, g.frame_bytes + 256));
        }
        if (scratch && !conv) {
            l.drawn = 2; /* the picture leaves from the overlay's own copy */
        }
        DrawItem *di = nullptr;
        if (l.drawn) {
            di = &draw[n_draw++];
            memset(di, 0, sizeof(*di));
            di->mvs = d_mv_ + (size_t) li * step_nblk;
            di->stab = d_stab_ + (size_t) li * step_nblk;
            di->blk_w = g.blk_w;
            di->blk_h = g.blk_h;
            di->nbh = g.nbh;
            di->nbv = g.nbv;
            di->mode = draw_mode;
        }
        for (int p = 0; p < 3 && want_out; p++) {
            uint8_t *F = nullptr;
            if (out[k].plane[p] && out[k].on_device && out[k].stride[p] == og.pw[p] && (dense_out || (!l.drawn && !conv))) {
                F = out[k].plane[p];
            } else if (out[k].plane[p] && hostp) {
                /* host destination, packed layout: pack on the device, one contiguous copy later */
                F = d_out_all_[step_no_ & 1] + out_pitch_ * li + og.plane_off[p];
            }
            /* N: dense picture in the stream's own format, the overlay's canvas */
            uint8_t *N = scratch ? l.d_draw + g.plane_off[p] : F;
            PlaneRef from = plane_ref(cur, p);
            if (l.drawn) {
                pack[n_pack].src = from;
                pack[n_pack].dst = N;
                n_pack++;
                di->dst[p] = N;
                di->stride[p] = g.pw[p];
                di->w[p] = g.pw[p];
                di->h[p] = g.ph[p];
                from.p = N;
                from.stride = g.pw[p];
                if (!conv) {
                    continue;
                }
            }
            if (!F) {
                continue;
            }
            if (conv && p > 0) {
                To420Item &t = cv[n_cv++];
                t.src = from;
                t.dst = F;
                t.dw = og.pw[p];
                t.dh = og.ph[p];
                t.hpass = g.subsamp == DSV_SUBSAMP_444;
            } else if (l.drawn) { /* luma of a drawn + converted picture: canvas -> destination */
                pack2[n_pack2].src = from;
                pack2[n_pack2].dst = F;
                n_pack2++;
            } else {
                pack[n_pack].src = from;
                pack[n_pack].dst = F;
                n_pack++;
            }
        }
        dec_bmc_fill(ba, &n_p, isP, motion_geom(g, 0), d_mv_, li, step_nblk, l.out[l.cur ^ 1], cur);
    }
    stats.host_ms += host_now_ms() - t_host0;
    if (n_sj == 0) {
        CUDA_CHECK(cudaStreamSynchronize(st));
        return;
    }
    const SbtDims sdims = sbt_assign_tiles(sj, n_sj);
    /* pictures of earlier steps may still be leaving on the copy stream: the frame buffers written now were read
     * by the copies of step t-2 (references alternate), or of step t-1 where that step had non-reference pictures */
    CUDA_CHECK(cudaStreamWaitEvent(st, ev_copied_[step_no_ & 1], 0));
    if (prev_nonref_) {
        CUDA_CHECK(cudaStreamWaitEvent(st, ev_copied_[(step_no_ ^ 1) & 1], 0));
    }
    {
        CopyItem up[3] = {{nullptr, nullptr, 0}, {d_stab_, h_stab_, (size_t) step_nblk * L_},
                          {d_mv_, h_mv_, n_p ? sizeof(DevMV) * (size_t) step_nblk * L_ : 0}};
        arena_.take_upload(&up[0]);
        copyn_launch(up, 3, st);
    }
    copy_launch(d_cpy, n_cpy, max_cpy, st);
    hzdec_clean_launch(d_clean, n_clean, g_.tiles[0], st);
    hzdec_launch_jobs(d_hzj, dims, st);
    sbt_inv_launch(d_sj, sdims, g_.lo_smem, st, timed ? ev_[0] : nullptr, timed ? ev_[1] : nullptr);
    if (n_p && timed) {
        CUDA_CHECK(cudaEventRecord(ev_[2], st));
    }
    bmc_launch(d_bmc, n_p, motion_geom(step_g, 0), st);
    if (n_p && timed) {
        CUDA_CHECK(cudaEventRecord(ev_[3], st));
    }
    extend_launch(d_ext, n_ext, g_.w, g_.h, st);
    pack_launch(d_pack, n_pack, g_.w, g_.h, st);
    overlay_launch(d_draw, n_draw, st);
    pack_launch(d_pack2, n_pack2, g_.w, g_.h, st);
    to420_launch(d_cv, n_cv, og_.pw[1], og_.ph[1], st);
    stats.kernel_launches += 13 + (n_p ? 1 : 0) + (n_ext ? 1 : 0) + (n_pack ? 1 : 0) + (n_draw ? 1 : 0) + (n_pack2 ? 1 : 0) + (n_cv ? 1 : 0);
    CUDA_CHECK(cudaEventRecord(ev_done_, st));
    CUDA_CHECK(cudaStreamWaitEvent(st_copy_, ev_done_, 0));
    bool nonref = false;
    {
        /* packed host destinations at a constant distance (the batch API): one strided copy for all lanes */
        bool uniform = n > 0;
        const ptrdiff_t delta = n > 1 && out[0].plane[0] && out[1].plane[0] ? out[1].plane[0] - out[0].plane[0] : (ptrdiff_t) og_.frame_bytes;
        for (int k = 0; k < n && uniform; k++) {
            uniform = lane_ids[k] == k && lanes_[(size_t) k].ok && host_packed(og_, out[k]) && out[k].plane[0] == out[0].plane[0] + delta * k;
        }
        uniform = uniform && delta >= (ptrdiff_t) og_.frame_bytes;
        uint8_t *stage = d_out_all_[step_no_ & 1];
        if (uniform) {
            CUDA_CHECK(cudaMemcpy2DAsync(out[0].plane[0], (size_t) delta, stage, out_pitch_, og_.frame_bytes, (size_t) n, cudaMemcpyDeviceToHost, st_copy_));
            stats.d2h_bytes += og_.frame_bytes * (size_t) n;
        }
        for (int k = 0; k < n; k++) {
            const int li = lane_ids[k];
            DecLane &l = lanes_[(size_t) li];
            if (!l.ok || l.noout) {
                continue;
            }
            nonref |= !l.is_ref || l.drawn == 2; /* the overlay's copy is single-buffered */
            if (uniform || !out[k].plane[0] || out[k].on_device) {
                if (out[k].on_device) { /* strided device destination (not handled by pack_kernel) */
                    const DevFrame &cur = l.out[l.cur];
                    const bool via_draw = l.drawn == 2;
                    for (int p = 0; p < 3; p++) {
                        if (!out[k].plane[p]) {
                            continue;
                        }
                        if (via_draw) {
                            CUDA_CHECK(cudaMemcpy2DAsync(out[k].plane[p], (size_t) out[k].stride[p], l.d_draw + g_.plane_off[p], (size_t) g_.pw[p],
                                                         (size_t) g_.pw[p], (size_t) g_.ph[p], cudaMemcpyDeviceToDevice, st_copy_));
                        } else if (out[k].stride[p] != og_.pw[p]) {
                            CUDA_CHECK(cudaMemcpy2DAsync(out[k].plane[p], (size_t) out[k].stride[p], cur.p[p], (size_t) cur.stride[p], (size_t) g_.pw[p],
                                                         (size_t) g_.ph[p], cudaMemcpyDeviceToDevice, st_copy_));
                        }
                    }
                }
                continue;
            }
            if (host_packed(og_, out[k])) {
                CUDA_CHECK(cudaMemcpyAsync(out[k].plane[0], stage + out_pitch_ * li, og_.frame_bytes, cudaMemcpyDeviceToHost, st_copy_));
            } else { /* strided host frame (dsv_dec): straight from the bordered frame, or from the overlay's copy */
                const DevFrame &cur = l.out[l.cur];
                for (int p = 0; p < 3; p++) {
                    const uint8_t *src = l.drawn == 2 ? l.d_draw + g_.plane_off[p] : cur.p[p];
                    const size_t sstride = l.drawn == 2 ? (size_t) g_.pw[p] : (size_t) cur.stride[p];
                    CUDA_CHECK(cudaMemcpy2DAsync(out[k].plane[p], (size_t) out[k].stride[p], src, sstride, (size_t) g_.pw[p],
                                                 (size_t) g_.ph[p], cudaMemcpyDeviceToHost, st_copy_));
                }
            }
            stats.d2h_bytes += og_.frame_bytes;
        }
    }
    CUDA_CHECK(cudaEventRecord(ev_copied_[step_no_ & 1], st_copy_));
    prev_nonref_ = nonref;
    step_no_++;
    /* no wait here: the caller parses the next packets while this step runs (see collect()) */
    CUDA_CHECK(cudaEventRecord(ev_end_[par], st));
    pending_[par].valid = true;
    pending_[par].timed = timed;
    pending_[par].pictures = n_sj / 3;
    pending_[par].p_pictures = n_p;
    for (int k = 0; k < n; k++) {
        DecLane &l = lanes_[(size_t) lane_ids[k]];
        if (l.ok && l.is_ref) {
            l.have_ref = 1;
            l.cur ^= 1;
        }
    }
}

} // namespace dsv

/* ---- public API: DSV_DECODER.ref (the reference keeps its DSV_IMAGE there) holds a one-lane engine ---- */

static DecEngine *dec_engine(DSV_DECODER *d) { return reinterpret_cast<DecEngine *>(d->ref); }

extern "C" DSV_META *dsv_get_metadata(DSV_DECODER *d)
{
    DSV_META *m = (DSV_META *) dsv_alloc(sizeof(DSV_META));
    *m = d->vidmeta;
    return m;
}

extern "C" void dsv_dec_free(DSV_DECODER *d)
{
    delete dec_engine(d);
    d->ref = NULL;
}

void dsv::parse_metadata_packet(const uint8_t *pkt, unsigned len, DSV_META *m) /* dsv_decoder.c:50-70 */
{
    BitReader br(pkt, len);
    br.skip_bytes(DSV_PACKET_HDR_SIZE);
    m->width = (int) br.get_ueg();
    m->height = (int) br.get_ueg();
    m->subsamp = (int) br.get_ueg();
    m->fps_num = (int) br.get_ueg();
    m->fps_den = (int) br.get_ueg();
    m->aspect_num = (int) br.get_ueg();
    m->aspect_den = (int) br.get_ueg();
}

extern "C" int dsv_dec(DSV_DECODER *d, DSV_BUF *buffer, DSV_FRAME **out, DSV_FNUM *fn)
{
    DSV_API_BEGIN
    *fn = (DSV_FNUM) -1;
    const uint8_t *pkt = buffer->data;
    const unsigned pkt_len = buffer->len;
    BitReader br(pkt, pkt_len);
    const int pkt_type = read_packet_hdr(br);
    if (pkt_type == -1) {
        dsv_buf_free(buffer);
        return DSV_DEC_ERROR;
    }
    if (!DSV_PT_IS_PIC(pkt_type)) {
        int ret = DSV_DEC_ERROR;
        if (pkt_type == DSV_PT_META) {
            parse_metadata_packet(pkt, pkt_len, &d->vidmeta);
            d->got_metadata = 1;
            ret = DSV_DEC_GOT_META;
        } else if (pkt_type == DSV_PT_EOS) {
            ret = DSV_DEC_EOS;
        }
        dsv_buf_free(buffer);
        return ret;
    }
    if (!d->got_metadata) {
        DSV_WARNING(("no metadata, skipping frame"));
        dsv_buf_free(buffer);
        return DSV_DEC_OK;
    }
    const DSV_META &md = d->vidmeta;
    if (!meta_supported(md)) {
        DSV_ERROR(("unsupported picture format %dx%d subsamp %d", md.width, md.height, md.subsamp));
        dsv_buf_free(buffer);
        return DSV_DEC_ERROR;
    }
    DecEngine *e = dec_engine(d);
    if (e && !e->matches(md)) {
        delete e; /* new sequence parameters: references of the old size are useless */
        e = nullptr;
    }
    if (!e) {
        e = new DecEngine(md, 1);
        d->ref = reinterpret_cast<DSV_IMAGE *>(e);
    }
    e->draw_mode = d->draw_info;
    DSV_FRAME *f = mk_frame_pinned(md.subsamp, md.width, md.height);
    PktRef pr = {pkt, nullptr, pkt_len};
    OutRef o;
    for (int p = 0; p < 3; p++) {
        o.plane[p] = f->planes[p].data;
        o.stride[p] = f->planes[p].stride;
    }
    o.on_device = 0;
    const int lane = 0;
    int code = DSV_DEC_ERROR;
    e->step(1, &lane, &pr, &o, &code, fn);
    e->flush();
    if (code != DSV_DEC_OK) {
        dsv_frame_ref_dec(f);
        /* the reference frees the packet on every error path except the missing-reference one
         * (dsv_decoder.c:356 vs 424-427) */
        if (*fn == (DSV_FNUM) -1) {
            dsv_buf_free(buffer);
        }
        return DSV_DEC_ERROR;
    }
    dsv_buf_free(buffer);
    *out = f;
    return DSV_DEC_OK;
    DSV_API_END(DSV_DEC_ERROR)
}
