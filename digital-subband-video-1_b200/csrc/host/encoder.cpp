/*
 * encoder.cpp -- the dsv_encoder.h API (dsv_encoder.c:696-854) and the lock-step encode engine behind it.
 *
 * Host code here does only what is serial and tiny in the reference: GOP / frame-type decisions
 * (dsv_encoder.c:575-694), the CRF quality->quant map (dsv_encoder.c:162-165), the ABR controller
 * (dsv_encoder.c:84-160,816-848), the stability tracker and its ZBRLE map (dsv_encoder.c:329-408),
 * motion-vector prediction + side-info sub-streams (dsv_encoder.c:256-327, dsv.c:189-231) and packet
 * framing (dsv_encoder.c:170-192,410-536).  Every per-pixel / per-coefficient / per-bit stage is a kernel
 * launch batched over all lanes of the engine, on the engine's stream:
 *   phase 1  ingest (+border) -> luma pyramid -> luma sum -> HME            [sync: MVs, sums, intra counts]
 *   phase 2  host: frame types, quantiser, stability map, motion side info -> packet heads
 *   phase 3  BMC + residual -> SBT forward + quantise -> HZCC scan/prefix/pack [event: packet sizes]
 *            -> SBT inverse -> reconstruction + border (new references) || packets D2H   [sync]
 * There is no CPU implementation of those stages in this library.
 */
#include <cmath>

#include "dsv1_b200.h"

#include "bits.h"
#include "engine.h"

using namespace dsv;

namespace dsv {

int size4dim(int dim) /* dsv_encoder.c:556-572 */
{
    if (dim > 1280) return 64;
    if (dim > 1024) return 48;
    if (dim > 704) return 32;
    if (dim > 352) return 24;
    return 16;
}

void plan_geometry(CodecGeom *g, int w, int h, int subsamp)
{
    memset(g, 0, sizeof(*g));
    g->w = w;
    g->h = h;
    g->subsamp = subsamp;
    g->hs = DSV_FORMAT_H_SHIFT(subsamp);
    g->vs = DSV_FORMAT_V_SHIFT(subsamp);
    g->pw[0] = w;
    g->ph[0] = h;
    g->pw[1] = g->pw[2] = ceil_shift(w, g->hs);
    g->ph[1] = g->ph[2] = ceil_shift(h, g->vs);
    g->cw[0] = w;
    g->ch[0] = h;
    g->cw[1] = g->cw[2] = (g->pw[1] + 1) & ~1; /* dsv_mk_coefs: chroma rounded up to even */
    g->ch[1] = g->ch[2] = (g->ph[1] + 1) & ~1;
    g->coef_off[0] = 0;
    g->coef_off[1] = (size_t) g->cw[0] * g->ch[0];
    g->coef_off[2] = g->coef_off[1] + (size_t) g->cw[1] * g->ch[1];
    g->coef_total = g->coef_off[2] + (size_t) g->cw[2] * g->ch[2];
    g->plane_off[0] = 0;
    g->plane_off[1] = (size_t) w * h;
    g->plane_off[2] = g->plane_off[1] + (size_t) g->pw[1] * g->ph[1];
    g->frame_bytes = g->plane_off[2] + (size_t) g->pw[2] * g->ph[2];
    g->lo_smem = 0;
    for (int p = 0; p < 3; p++) {
        g->tiles[p] = ceil_div(g->cw[p], SBT_TW) * ceil_div(g->ch[p], SBT_TH);
        g->total_tiles += g->tiles[p];
        HzRegions r;
        hz_fill_regions(&r, g->cw[p], g->ch[p]);
        g->chunks[p] = ceil_div(r.base[HZ_NREG], HZ_CHUNK);
        g->total_chunks += g->chunks[p];
        size_t s = sbt_lo_smem_bytes(g->cw[p], g->ch[p]);
        g->lo_smem = s > g->lo_smem ? s : g->lo_smem;
    }
}

void plan_blocks(CodecGeom *g, int blk_w, int blk_h)
{
    g->blk_w = blk_w;
    g->blk_h = blk_h;
    g->nbh = ceil_div(g->w, blk_w);
    g->nbv = ceil_div(g->h, blk_h);
    g->nblk = g->nbh * g->nbv;
}

MotionGeom motion_geom(const CodecGeom &g, int levels)
{
    return {g.w, g.h, g.hs, g.vs, g.blk_w, g.blk_h, g.nbh, g.nbv, levels};
}

bool meta_supported(const DSV_META &m)
{
    if (m.width < 16 || m.height < 16 || (m.width & 1) || (m.height & 1) || m.width > 16384 || m.height > 16384) {
        return false;
    }
    return m.subsamp == DSV_SUBSAMP_444 || m.subsamp == DSV_SUBSAMP_422 || m.subsamp == DSV_SUBSAMP_420 ||
           m.subsamp == DSV_SUBSAMP_411;
}

} // namespace dsv

/* ---- packet pieces -------------------------------------------------------------------------- */

static void put_packet_hdr(BitWriter &bw, int pkt_type) /* dsv_encoder.c:410-424 */
{
    bw.put_bits(8, DSV_FOURCC_0);
    bw.put_bits(8, DSV_FOURCC_1);
    bw.put_bits(8, DSV_FOURCC_2);
    bw.put_bits(8, DSV_FOURCC_3);
    bw.put_bits(8, DSV_VERSION_MINOR);
    bw.put_bits(8, (uint32_t) pkt_type);
    bw.put_bits(32, 0);
    bw.put_bits(32, 0);
}

static void put_be32(uint8_t *p, unsigned v)
{
    p[0] = (uint8_t) (v >> 24);
    p[1] = (uint8_t) (v >> 16);
    p[2] = (uint8_t) (v >> 8);
    p[3] = (uint8_t) v;
}

static void set_links(DSV_ENCODER *enc, DSV_BUF *buf, int is_eos) /* dsv_encoder.c:170-192 */
{
    unsigned next = is_eos ? 0 : buf->len;
    put_be32(buf->data + DSV_PACKET_PREV_OFFSET, (unsigned) enc->prev_link);
    put_be32(buf->data + DSV_PACKET_NEXT_OFFSET, next);
    enc->prev_link = (int) next;
}

void dsv::make_metadata_packet(DSV_ENCODER *enc, DSV_BUF *buf) /* dsv_encoder.c:426-461 */
{
    const DSV_META &m = enc->vidmeta;
    dsv_mk_buf(buf, 64);
    BitWriter bw(buf->data);
    put_packet_hdr(bw, DSV_PT_META);
    bw.put_ueg((uint32_t) m.width);
    bw.put_ueg((uint32_t) m.height);
    bw.put_ueg((uint32_t) m.subsamp);
    bw.put_ueg((uint32_t) m.fps_num);
    bw.put_ueg((uint32_t) m.fps_den);
    bw.put_ueg((uint32_t) m.aspect_num);
    bw.put_ueg((uint32_t) m.aspect_den);
    bw.align();
    buf->len = bw.byte_pos();
    put_be32(buf->data + DSV_PACKET_NEXT_OFFSET, buf->len);
}

/* stability tracker + its ZBRLE map (dsv_encoder.c:329-408); also fills enc->stable_blocks */
static void put_stable_blocks(DSV_ENCODER *enc, const CodecGeom &g, int isP, const DevMV *mvs, BitWriter &bw)
{
    const int nblk = g.nblk;
    std::vector<uint8_t> tmp((size_t) nblk + 64, 0); /* ZBRLE: at most ~1 bit per block plus the final run */
    RleWriter rle(tmp.data());
    if (enc->refresh_ctr >= enc->stable_refresh) {
        enc->refresh_ctr = 0;
        memset(enc->stability, 0, sizeof(*enc->stability) * (size_t) nblk);
    }
    int avgdiv = (int) enc->refresh_ctr;
    if (avgdiv <= 0) {
        avgdiv = 1;
    }
    for (int i = 0; i < nblk; i++) {
        int stable = 0, intra = 0;
        if (isP) {
            const DevMV &mv = mvs[i];
            if (mv.mode == DSV_MODE_INTER) {
                enc->stability[i].x += iabs(mv.x) >> 2;
                enc->stability[i].y += iabs(mv.y) >> 2;
                stable = mv.high_detail;
                int ax = enc->stability[i].x / avgdiv, ay = enc->stability[i].y / avgdiv;
                stable |= (ax == 0 && ay == 0 && !mv.lo_tex && !mv.lo_var);
            } else {
                intra = 1;
            }
            if (mv.lo_tex || mv.lo_var) { /* not worth bits: poison the accumulators */
                enc->stability[i].x = 0x3fff;
                enc->stability[i].y = 0x3fff;
            }
        } else {
            int ax = enc->stability[i].x / avgdiv, ay = enc->stability[i].y / avgdiv;
            stable = (ax == 0 && ay == 0);
        }
        enc->stable_blocks[i] = (unsigned char) (stable | (intra << 1));
        rle.put(stable & 1);
    }
    bw.align();
    unsigned bytes = rle.finish();
    bw.put_ueg(bytes);
    bw.align();
    bw.concat(tmp.data(), bytes);
}

static int mv_pred1(int left, int top, int topleft) /* dsv.c:189-197 */
{
    int dif = left + top - topleft;
    return iabs(dif - left) < iabs(dif - top) ? left : top;
}

void dsv::predict_mv(const DevMV *mvs, int nbh, int x, int y, int *px, int *py) /* dsv.c:199-231 */
{
    int vx[3] = {0, 0, 0}, vy[3] = {0, 0, 0};
    if (x > 0) {
        const DevMV &m = mvs[y * nbh + x - 1];
        if (m.mode == DSV_MODE_INTER) { vx[0] = m.x; vy[0] = m.y; }
    }
    if (y > 0) {
        const DevMV &m = mvs[(y - 1) * nbh + x];
        if (m.mode == DSV_MODE_INTER) { vx[1] = m.x; vy[1] = m.y; }
    }
    if (x > 0 && y > 0) {
        const DevMV &m = mvs[(y - 1) * nbh + x - 1];
        if (m.mode == DSV_MODE_INTER) { vx[2] = m.x; vy[2] = m.y; }
    }
    *px = mv_pred1(vx[0], vx[1], vx[2]);
    *py = mv_pred1(vy[0], vy[1], vy[2]);
}

/* four byte-aligned sub-streams: modes (ZBRLE), MV x, MV y (SEG of prediction error), intra masks
 * (dsv_encoder.c:256-327) */
static void put_motion(const CodecGeom &g, const DevMV *mvs, BitWriter &bw)
{
    const int nbh = g.nbh, nbv = g.nbv;
    /* worst case per block: 1-2 bits of mode run, SEG of a 16-bit delta (34 bits), 5 mask bits */
    const size_t ub = (size_t) nbh * nbv * 6 + 64;
    std::vector<uint8_t> b_mode(ub, 0), b_x(ub, 0), b_y(ub, 0), b_mask(ub, 0);
    RleWriter rle(b_mode.data());
    BitWriter wx(b_x.data()), wy(b_y.data()), wm(b_mask.data());
    for (int j = 0; j < nbv; j++) {
        for (int i = 0; i < nbh; i++) {
            const DevMV &mv = mvs[j * nbh + i];
            rle.put(mv.mode);
            if (mv.mode == DSV_MODE_INTER) {
                int px, py;
                predict_mv(mvs, nbh, i, j, &px, &py);
                wx.put_seg(mv.x - px);
                wy.put_seg(mv.y - py);
            } else if (mv.submask == DSV_MASK_ALL_INTRA) {
                wm.put_bit(1);
            } else {
                wm.put_bit(0);
                wm.put_bits(4, mv.submask);
            }
        }
    }
    unsigned n_mode = rle.finish();
    wx.align();
    wy.align();
    wm.align();
    const uint8_t *data[4] = {b_mode.data(), b_x.data(), b_y.data(), b_mask.data()};
    unsigned len[4] = {n_mode, wx.byte_pos(), wy.byte_pos(), wm.byte_pos()};
    for (int s = 0; s < 4; s++) {
        bw.align();
        bw.put_ueg(len[s]);
        bw.align();
        bw.concat(data[s], len[s]);
    }
}

/* ABR controller (dsv_encoder.c:84-160): host-only, needs every previous packet's size, hence 1 GPU */
static int rate_control_quality(DSV_ENCODER *enc, int isP, int forced_intra)
{
    int q = (int) enc->rc_quant;
    if (enc->rc_mode == DSV_RATE_CONTROL_CRF) {
        q = enc->quality;
        enc->rc_quant = (unsigned) q;
        return q;
    }
    const DSV_META &vf = enc->vidmeta;
    int fps = (vf.fps_num << 5) / vf.fps_den;
    if (fps == 0) {
        fps = 1;
    }
    int needed_bpf = (int) (((enc->bitrate << 5) / (unsigned) fps) >> 3);
    int bpf = enc->bpf_avg ? enc->bpf_avg : needed_bpf;
    int dir = (bpf - needed_bpf) > 0 ? -1 : 1;
    int delta = (iabs(bpf - needed_bpf) << 9) / needed_bpf;
    int nudged = 0;
    if (dir == 1) {
        delta *= 2;
    }
    if (enc->rc_high_motion_nudge) {
        if (isP && enc->last_P_frame_over) {
            delta = (delta + 1) * 2;
            dir = -1;
            nudged = 1;
        } else if (enc->back_into_range) {
            delta = (delta + 1) * 2;
            dir = 1;
            nudged = 1;
        }
    }
    delta = (q * delta) >> 9;
    enc->max_q_step = iclamp(enc->max_q_step, 1, DSV_MAX_QUALITY);
    delta = imin(delta, nudged ? enc->max_q_step * 16 : enc->max_q_step);
    q += delta * dir;
    int low_p = iclamp(enc->avg_P_frame_q - DSV_QUALITY_PERCENT(4), enc->min_quality, enc->max_quality);
    int minq = isP ? low_p : enc->min_I_frame_quality;
    if (forced_intra) {
        if (q < DSV_QUALITY_PERCENT(60)) {
            q += DSV_QUALITY_PERCENT(15);
        } else if (q < DSV_QUALITY_PERCENT(70)) {
            q += DSV_QUALITY_PERCENT(8);
        } else if (q < DSV_QUALITY_PERCENT(75)) {
            q += DSV_QUALITY_PERCENT(3);
        }
        q = iclamp(q, 0, enc->max_quality - DSV_QUALITY_PERCENT(5));
    }
    q = iclamp(q, minq, enc->max_quality);
    q = iclamp(q, 0, DSV_MAX_QUALITY);
    enc->rc_quant = (unsigned) q;
    return q;
}

static void rate_control_update(DSV_ENCODER *enc, int isP, unsigned pkt_len) /* dsv_encoder.c:816-848 */
{
    if (enc->rc_mode == DSV_RATE_CONTROL_CRF) {
        return;
    }
    enc->bpf_total += pkt_len;
    enc->bpf_reset++;
    if (isP) {
        enc->total_P_frame_q += (int) enc->rc_quant;
        enc->avg_P_frame_q = enc->total_P_frame_q / (int) enc->bpf_reset;
        unsigned fps = (unsigned) ((enc->vidmeta.fps_num << 5) / enc->vidmeta.fps_den);
        if (fps == 0) {
            fps = 1;
        }
        unsigned needed = ((enc->bitrate << 5) / fps) >> 3;
        int under = pkt_len < (needed * 3 / 4);
        int over = pkt_len > (needed * 7 / 8);
        enc->back_into_range = (enc->last_P_frame_over && under);
        enc->last_P_frame_over = over;
    } else {
        enc->last_P_frame_over = 0;
        enc->back_into_range = 0;
    }
    enc->bpf_avg = (int) (enc->bpf_total / enc->bpf_reset);
    if (enc->bpf_reset >= DSV_BPF_RESET) {
        enc->bpf_total = (unsigned) enc->bpf_avg;
        enc->total_P_frame_q = enc->total_P_frame_q / (int) enc->bpf_reset;
        enc->bpf_reset = 1;
    }
}


/* ============================================================================================== */
/* lock-step encode engine                                                                        */
/* ============================================================================================== */

namespace dsv {

EncEngine::EncEngine(const DSV_META &md, int gop, int pyramid_levels, int lanes)
{
    if (!meta_supported(md)) {
        DSV_ERROR(("unsupported picture format %dx%d subsamp %d: width and height must be even and >= 16", md.width,
                   md.height, md.subsamp));
        throw Unsupported();
    }
    CUDA_CHECK(cudaGetDevice(&device));
    plan_geometry(&g_, md.width, md.height, md.subsamp);
    plan_blocks(&g_, iclamp(size4dim(md.width) & ~7, DSV_MIN_BLOCK_SIZE, DSV_MAX_BLOCK_SIZE),
                iclamp(size4dim(md.height) & ~7, DSV_MIN_BLOCK_SIZE, DSV_MAX_BLOCK_SIZE));
    inter_ = gop != DSV_GOP_INTRA;
    levels_ = pyramid_levels;
    L_ = lanes;
    if (const char *e = getenv("DSV_KERNEL_TIMES")) {
        time_kernels = atoi(e) != 0;
    }
    CUDA_CHECK(cudaStreamCreateWithFlags(&st_, cudaStreamNonBlocking));
    CUDA_CHECK(cudaStreamCreateWithFlags(&st_copy_, cudaStreamNonBlocking));
    for (auto &e : ev_) {
        CUDA_CHECK(cudaEventCreate(&e));
    }
    CUDA_CHECK(cudaEventCreateWithFlags(&ev_search_, cudaEventDisableTiming));
    CUDA_CHECK(cudaEventCreateWithFlags(&ev_sizes_, cudaEventDisableTiming));
    for (auto &e : ev_pref_) {
        CUDA_CHECK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    }
    const size_t per_lane = 3 * (sizeof(SbtJob) + sizeof(HzJob)) + sizeof(HzFrame) + (size_t) (levels_ + 1) * sizeof(HmeArgs) +
                            sizeof(BmcArgs) + 8 * sizeof(PlaneRef) + 2 * sizeof(ZeroItem) + 2048;
    arena_.create(per_lane * (size_t) L_ + 4096);
    CUDA_CHECK(cudaMalloc(&d_mv0_, sizeof(DevMV) * (size_t) g_.nblk * L_));
    CUDA_CHECK(cudaMemset(d_mv0_, 0, sizeof(DevMV) * (size_t) g_.nblk * L_));
    CUDA_CHECK(cudaMallocHost(&h_mv0_, sizeof(DevMV) * (size_t) g_.nblk * L_));
    memset(h_mv0_, 0, sizeof(DevMV) * (size_t) g_.nblk * L_);
    CUDA_CHECK(cudaMalloc(&d_stab_, (size_t) g_.nblk * L_));
    CUDA_CHECK(cudaMallocHost(&h_stab_, (size_t) g_.nblk * L_));
    CUDA_CHECK(cudaMalloc(&d_misc_, sizeof(LaneMisc) * (size_t) L_));
    CUDA_CHECK(cudaMallocHost(&h_misc_, sizeof(LaneMisc) * (size_t) L_));
    CUDA_CHECK(cudaMalloc(&d_chunks_, sizeof(HzChunk) * (size_t) g_.total_chunks * L_));
    CUDA_CHECK(cudaMalloc(&d_frames_, sizeof(HzFrame) * (size_t) L_));
    CUDA_CHECK(cudaMallocHost(&h_frames_, sizeof(HzFrame) * (size_t) L_));
    CUDA_CHECK(cudaMallocHost(&h_pk_, sizeof(CopyItem) * (size_t) L_));
    in_pitch_ = (g_.frame_bytes + 255) & ~(size_t) 255;
    for (auto &b : d_in_all_) {
        CUDA_CHECK(cudaMalloc(&b, in_pitch_ * L_ + 256));
    }
    if (L_ > 1) {
        int nt = (int) std::thread::hardware_concurrency() / 2;
        if (const char *e = getenv("DSV_HOST_THREADS")) {
            nt = atoi(e);
        }
        nt = iclamp(nt, 1, 8);
        pool_ = new HostPool(nt - 1); /* the calling thread works too */
    }
    lanes_.resize((size_t) L_);
    for (int i = 0; i < L_; i++) {
        enc_lane_alloc(lanes_[(size_t) i], g_, inter_, levels_, enc_packet_cap(g_));
        lanes_[(size_t) i].d_mvf[0] = d_mv0_ + (size_t) i * g_.nblk;
        for (int b = 0; b < ENC_STAGE_SLOTS; b++) {
            lanes_[(size_t) i].d_in[b] = d_in_all_[b] + in_pitch_ * i;
        }
    }
}

EncEngine::~EncEngine()
{
    cudaStreamSynchronize(st_);
    delete pool_;
    for (auto &l : lanes_) {
        enc_lane_free(l);
    }
    arena_.destroy();
    for (auto &b : d_in_all_) {
        cudaFree(b);
    }
    cudaFree(d_mv0_);
    cudaFreeHost(h_mv0_);
    cudaFree(d_stab_);
    cudaFreeHost(h_stab_);
    cudaFree(d_misc_);
    cudaFreeHost(h_misc_);
    cudaFree(d_chunks_);
    cudaFree(d_frames_);
    cudaFreeHost(h_frames_);
    cudaFreeHost(h_pk_);
    cudaFree(d_sse_);
    cudaFreeHost(h_sse_);
    cudaFree(d_ssim_);
    cudaFreeHost(h_ssim_);
    for (auto &e : ev_) {
        cudaEventDestroy(e);
    }
    ktimes.destroy();
    cudaEventDestroy(ev_search_);
    cudaEventDestroy(ev_sizes_);
    for (auto &e : ev_pref_) {
        cudaEventDestroy(e);
    }
    cudaStreamDestroy(st_copy_);
    cudaStreamDestroy(st_);
}

/* The per-picture reports' buffers, made when a step first runs with a report on whose buffers do not exist yet (no
 * step is in flight then: step() ends with a stream synchronisation): per report the sums, the step arena and packet
 * copy list grown by its jobs, its zero item and its sums' copy item; with the first report, for intra-only engines,
 * a reconstruction target per lane (their inverse would write in place over the source). */
void EncEngine::enable_reports(bool sse, bool ssim)
{
    const size_t sums = (sizeof(unsigned long long) * 3 * (size_t) L_ + 15) & ~(size_t) 15;
    const size_t per_report = (3 * sizeof(SseJob) + 16) * (size_t) L_ + sizeof(ZeroItem) + 64;
    const bool add_sse = sse && !d_sse_, add_ssim = ssim && !d_ssim_, first = !d_sse_ && !d_ssim_;
    const size_t arena = arena_.cap + per_report * (size_t) ((add_sse ? 1 : 0) + (add_ssim ? 1 : 0));
    arena_.destroy();
    arena_.create(arena);
    if (add_sse) {
        CUDA_CHECK(cudaMalloc(&d_sse_, sums));
        CUDA_CHECK(cudaMallocHost(&h_sse_, sums));
    }
    if (add_ssim) {
        CUDA_CHECK(cudaMalloc(&d_ssim_, sums));
        CUDA_CHECK(cudaMallocHost(&h_ssim_, sums));
    }
    cudaFreeHost(h_pk_);
    h_pk_ = nullptr;
    CUDA_CHECK(cudaMallocHost(&h_pk_, sizeof(CopyItem) * ((size_t) L_ + (d_sse_ ? 1 : 0) + (d_ssim_ ? 1 : 0))));
    if (!inter_ && first) {
        for (auto &l : lanes_) {
            devframe_alloc(&l.qrec, g_.w, g_.h, g_.subsamp);
        }
    }
}

static bool packed_pic(const CodecGeom &g, const PicRef &r)
{
    return r.stride[0] == g.pw[0] && r.stride[1] == g.pw[1] && r.stride[2] == g.pw[2] &&
           r.plane[1] == r.plane[0] + g.plane_off[1] && r.plane[2] == r.plane[0] + g.plane_off[2];
}

void EncEngine::prefetch(int n, const int *lane_ids, const PicRef *src)
{
    const CodecGeom &g = g_;
    bool used[ENC_STAGE_SLOTS] = {};
    /* common case (the batch API): lanes 0..n-1, packed pictures at a constant distance from each other and all
     * lanes on the same staging parity -> ONE strided copy for the whole step instead of 3n API calls */
    bool uniform = n > 0 && !src[0].on_device;
    const ptrdiff_t delta = n > 1 ? src[1].plane[0] - src[0].plane[0] : (ptrdiff_t) g.frame_bytes;
    for (int k = 0; k < n && uniform; k++) {
        uniform = lane_ids[k] == k && !src[k].on_device && packed_pic(g, src[k]) && lanes_[(size_t) k].in_sel == lanes_[0].in_sel &&
                  src[k].plane[0] == src[0].plane[0] + delta * k;
    }
    if (uniform && delta >= (ptrdiff_t) g.frame_bytes) {
        const int b = lanes_[0].in_sel;
        CUDA_CHECK(cudaMemcpy2DAsync(d_in_all_[b], in_pitch_, src[0].plane[0], (size_t) delta, g.frame_bytes, (size_t) n, cudaMemcpyHostToDevice, st_copy_));
        stats.h2d_bytes += g.frame_bytes * (size_t) n;
        for (int k = 0; k < n; k++) {
            EncLane &l = lanes_[(size_t) k];
            l.stage_src[b] = src[k].plane[0];
            l.in_sel = (l.in_sel + 1) % ENC_STAGE_SLOTS;
        }
        CUDA_CHECK(cudaEventRecord(ev_pref_[b], st_copy_));
        return;
    }
    for (int k = 0; k < n; k++) {
        EncLane &l = lanes_[(size_t) lane_ids[k]];
        if (src[k].on_device) {
            continue;
        }
        const int b = l.in_sel;
        uint8_t *buf = l.d_in[b];
        if (packed_pic(g, src[k])) {
            CUDA_CHECK(cudaMemcpyAsync(buf, src[k].plane[0], g.frame_bytes, cudaMemcpyHostToDevice, st_copy_));
        } else {
            for (int p = 0; p < 3; p++) {
                CUDA_CHECK(cudaMemcpy2DAsync(buf + g.plane_off[p], (size_t) g.pw[p], src[k].plane[p], (size_t) src[k].stride[p], (size_t) g.pw[p],
                                             (size_t) g.ph[p], cudaMemcpyHostToDevice, st_copy_));
            }
        }
        stats.h2d_bytes += g.frame_bytes;
        l.stage_src[b] = src[k].plane[0];
        l.in_sel = (l.in_sel + 1) % ENC_STAGE_SLOTS;
        used[b] = true;
    }
    for (int b = 0; b < ENC_STAGE_SLOTS; b++) {
        if (used[b]) {
            CUDA_CHECK(cudaEventRecord(ev_pref_[b], st_copy_));
        }
    }
}

void gop_bookkeeping(DSV_ENCODER *enc, bool inter, DSV_FNUM fnum, int *gop_start, int *is_ref, int *has_ref)
{
    *gop_start = 0;
    *is_ref = *has_ref = 0;
    if (enc->force_metadata || ((enc->prev_gop + (DSV_FNUM) enc->gop) <= fnum)) {
        *gop_start = 1;
        enc->prev_gop = fnum;
        enc->force_metadata = 0;
    }
    if (inter) {
        *is_ref = 1;
        *has_ref = !*gop_start;
    }
}

void decide_and_head(DSV_ENCODER *enc, const CodecGeom &g, bool inter, int top_samples, unsigned long long luma_sum, int nintra,
                     const DevMV *mvs, DSV_FNUM fnum, int is_ref, int *has_ref, int *forced_intra, int *quant, uint8_t *head,
                     unsigned *head_bytes)
{
    if (inter) {
        if (enc->do_scd) { /* check_scene_change, dsv_encoder.c:538-554 */
            int al = (int) (luma_sum / (unsigned long long) top_samples);
            if (iabs(enc->prev_avg_luma - al) > enc->scene_change_delta) {
                *has_ref = 0;
                *forced_intra = 1;
            }
            enc->prev_avg_luma = al;
        }
        if (*has_ref) { /* motion_est's verdict, dsv_encoder.c:246-253 */
            int pct = nintra * 100 / g.nblk;
            *forced_intra = 0;
            if (pct > enc->intra_pct_thresh) {
                *has_ref = 0;
                *forced_intra = 1;
            }
        }
    }
    const int isP = *has_ref;
    const int quality = rate_control_quality(enc, isP, *forced_intra);
    *quant = DSV_MAX_QUALITY - ((DSV_MAX_QUALITY - 5) * quality / DSV_MAX_QUALITY); /* dsv_encoder.c:165 */

    memset(head, 0, 256 + (size_t) g.nblk * 12); /* head <= 20 + stability map + 4 motion sub-streams (<= ~10 B per block) */
    BitWriter bw(head);
    put_packet_hdr(bw, DSV_MAKE_PT(is_ref, *has_ref));
    bw.align();
    bw.put_bits(32, fnum);
    bw.align();
    bw.put_ueg((uint32_t) (g.blk_w >> 2));
    bw.put_ueg((uint32_t) (g.blk_h >> 2));
    bw.align();
    put_stable_blocks(enc, g, isP, mvs, bw);
    if (isP) {
        bw.align();
        put_motion(g, mvs, bw);
    }
    bw.align();
    bw.put_bits(DSV_MAX_QP_BITS, (uint32_t) *quant);
    bw.align(); /* dsv_encode_plane aligns before each plane (hzcc.c:457) */
    *head_bytes = bw.byte_pos();
}

void EncEngine::step(int n, const int *lane_ids, const PicRef *src, DSV_BUF (*bufs)[2], int *nbufs, PktSink *sinks, const LongPlan *plan)
{
    const bool analyse = plan && plan[0].analyse, code = plan && !plan[0].analyse;
    const CodecGeom &g = g_;
    cudaStream_t st = st_;
    const MotionGeom mg = motion_geom(g, levels_);
    LaneMisc *h_misc = reinterpret_cast<LaneMisc *>(h_misc_), *d_misc = reinterpret_cast<LaneMisc *>(d_misc_);
    const bool timed = time_kernels;
    KtActivate kt_on(timed ? &ktimes : nullptr);
    ktimes.open(0);
    const bool sse_on = picture_info && !analyse, ssim_on = picture_ssim && !analyse;
    const bool report = sse_on || ssim_on; /* a report measures the reconstruction: every picture gets one */
    if ((sse_on && !d_sse_) || (ssim_on && !d_ssim_)) {
        enable_reports(sse_on, ssim_on);
    }
    arena_.reset();

    /* ---- phase 1: ingest, pyramid, luma sums, motion search -------------------------------------- */
    IngestItem *d_ing;
    IngestItem *ing = arena_.push_n<IngestItem>((size_t) 3 * n, &d_ing);
    bool wait_pref[ENC_STAGE_SLOTS] = {};
    for (int k = 0; k < n; k++) {
        EncLane &l = lanes_[(size_t) lane_ids[k]];
        l.fnum = plan ? plan[k].fnum : l.enc->next_fnum++;
        const DevFrame &dst = inter_ ? l.pad[l.cur] : l.xf;
        int pb = -1;
        if (!src[k].on_device) {
            for (int b = 0; b < ENC_STAGE_SLOTS && pb < 0; b++) {
                pb = l.stage_src[b] == src[k].plane[0] ? b : -1;
            }
        }
        const bool prefetched = pb >= 0;
        if (prefetched) {
            wait_pref[pb] = true;
            l.stage_src[pb] = nullptr;
        }
        uint8_t *stage_buf = prefetched ? l.d_in[pb] : l.d_in[l.in_sel];
        bool staged = false;
        const uint8_t *packed[3];
        for (int p = 0; p < 3; p++) {
            const size_t pbytes = (size_t) g.pw[p] * g.ph[p];
            if (src[k].on_device && src[k].stride[p] == g.pw[p]) {
                packed[p] = src[k].plane[p];
            } else if (prefetched) {
                packed[p] = stage_buf + g.plane_off[p];
            } else {
                uint8_t *stage = stage_buf + g.plane_off[p];
                CUDA_CHECK(cudaMemcpy2DAsync(stage, (size_t) g.pw[p], src[k].plane[p], (size_t) src[k].stride[p], (size_t) g.pw[p],
                                             (size_t) g.ph[p], src[k].on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st));
                if (!src[k].on_device) {
                    stats.h2d_bytes += pbytes;
                }
                packed[p] = stage;
                staged = true;
            }
        }
        ingest_fill_picture(&ing[3 * k], packed, dst);
        if (staged) {
            l.stage_src[l.in_sel] = nullptr;
            l.in_sel = (l.in_sel + 1) % ENC_STAGE_SLOTS;
        }
    }
    for (int b = 0; b < ENC_STAGE_SLOTS; b++) {
        if (wait_pref[b]) {
            CUDA_CHECK(cudaStreamWaitEvent(st, ev_pref_[b], 0));
        }
    }
    /* GOP bookkeeping (dsv_encoder.c:624-652): host state only */
    int n_search = 0, n_sum = 0;
    for (int k = 0; k < n; k++) {
        EncLane &l = lanes_[(size_t) lane_ids[k]];
        DSV_ENCODER *enc = l.enc;
        l.forced_intra = 0;
        if (plan) { /* metadata packets of a sharded sequence are written by the gather */
            l.gop_start = 0;
            l.is_ref = analyse ? 1 : plan[k].is_ref;
            l.has_ref = analyse ? (plan[k].search && l.have_ref) : plan[k].has_ref;
        } else {
            gop_bookkeeping(enc, inter_, l.fnum, &l.gop_start, &l.is_ref, &l.has_ref);
        }
        if (inter_) {
            if (l.has_ref && !l.have_ref) {
                DSV_ASSERT(0 && "P frame without a reference");
            }
            n_search += l.has_ref;
            n_sum += (analyse || (!plan && enc->do_scd)) ? 1 : 0;
        }
    }
    Down2Item *d_dn[DSV_MAX_PYRAMID_LEVELS] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    SumItem *d_sum = nullptr;
    HmeArgs *d_hme = nullptr;
    if (inter_ && !code) {
        for (int lv = 0; lv < levels_; lv++) {
            Down2Item *dn = arena_.push_n<Down2Item>((size_t) n, &d_dn[lv]);
            for (int k = 0; k < n; k++) {
                EncLane &l = lanes_[(size_t) lane_ids[k]];
                down2_fill_level(&dn[k], l.pad[l.cur], l.pyr[l.cur], lv);
            }
        }
        if (n_sum) {
            SumItem *sm = arena_.push_n<SumItem>((size_t) n_sum, &d_sum);
            int q = 0;
            for (int k = 0; k < n; k++) {
                EncLane &l = lanes_[(size_t) lane_ids[k]];
                if (analyse || l.enc->do_scd) {
                    sum_fill_lane(&sm[q++], l.pyr[l.cur], levels_, d_misc, lane_ids[k]);
                }
            }
        }
        if (n_search) { /* speculative: a scene change below simply discards the vectors */
            HmeArgs *ha = arena_.push_n<HmeArgs>((size_t) (levels_ + 1) * n_search, &d_hme);
            int q = 0;
            for (int k = 0; k < n; k++) {
                EncLane &l = lanes_[(size_t) lane_ids[k]];
                if (!l.has_ref) {
                    continue;
                }
                hme_fill_lane(ha, n_search, q++, mg, l.pad[l.cur], l.pyr[l.cur], l.pad[l.cur ^ 1], l.pyr[l.cur ^ 1], l.d_mvf, l.d_aux, d_misc,
                              lane_ids[k]);
            }
        }
    }
    /* motion compensation is launched right behind the search, before the host has seen the vectors: it depends on
     * nothing the host decides except "this stays a P picture", and when a scene change or the intra share turns
     * the picture into an I picture its output (prediction + residual frames) is simply not used.  The GPU works
     * on it while the host writes the packet heads. */
    BmcArgs *d_bmc = nullptr;
    if (n_search && !analyse) {
        BmcArgs *ba = arena_.push_n<BmcArgs>((size_t) n_search, &d_bmc);
        int q = 0;
        for (int k = 0; k < n; k++) {
            EncLane &l = lanes_[(size_t) lane_ids[k]];
            if (l.has_ref) {
                enc_bmc_fill(&ba[q++], mg, l.d_mvf[0], l.recon[l.cur ^ 1], l.pred, l.pad[l.cur], l.xf);
            }
        }
    }
    ZeroItem *d_zmisc;
    ZeroItem *zmisc = arena_.push_n<ZeroItem>(1, &d_zmisc);
    zmisc->p = d_misc_;
    zmisc->bytes = sizeof(LaneMisc) * (size_t) L_;
    arena_.upload(st);
    ingest_launch(d_ing, 3 * n, g.w, g.h, st);
    stats.kernel_launches += 1;
    bool need_sync = false;
    if (code && n_search) { /* the vectors found by the analysis pass */
        for (int k = 0; k < n; k++) {
            if (plan[k].has_ref) {
                memcpy(h_mv0_ + (size_t) lane_ids[k] * g.nblk, plan[k].mvs, sizeof(DevMV) * (size_t) g.nblk);
            }
        }
        copy1_launch(d_mv0_, h_mv0_, sizeof(DevMV) * (size_t) g.nblk * L_, st);
        if (timed) {
            CUDA_CHECK(cudaEventRecord(ev_[5], st));
        }
        bmc_launch(d_bmc, n_search, mg, st);
        if (timed) {
            CUDA_CHECK(cudaEventRecord(ev_[6], st));
        }
        stats.kernel_launches += 2;
    }
    if (inter_ && !code) {
        for (int lv = 0; lv < levels_; lv++) {
            down2_launch(d_dn[lv], n, ceil_shift(g.w, lv + 1), ceil_shift(g.h, lv + 1), st);
        }
        stats.kernel_launches += (unsigned) levels_;
        if (n_sum || n_search) {
            zero_launch(d_zmisc, 1, sizeof(LaneMisc) * (size_t) L_, st);
        }
        if (n_sum) {
            sum_launch(d_sum, n_sum, ceil_shift(g.h, levels_), st);
            stats.kernel_launches += 1;
        }
        if (n_search) {
            hme_launch(d_hme, n_search, mg, st);
            stats.kernel_launches += (unsigned) levels_ + 2;
        }
        if (n_sum || n_search) { /* the vectors and the per-lane sums come back in one launch */
            const CopyItem back[2] = {{h_mv0_, d_mv0_, n_search ? sizeof(DevMV) * (size_t) g.nblk * L_ : 0},
                                      {h_misc_, d_misc_, sizeof(LaneMisc) * (size_t) L_}};
            copyn_launch(back, 2, st);
            need_sync = true;
            CUDA_CHECK(cudaEventRecord(ev_search_, st));
        }
        if (n_search && !analyse) {
            if (timed) {
                CUDA_CHECK(cudaEventRecord(ev_[5], st));
            }
            bmc_launch(d_bmc, n_search, mg, st);
            if (timed) {
                CUDA_CHECK(cudaEventRecord(ev_[6], st));
            }
            stats.kernel_launches += 1;
        }
    }
    if (need_sync) {
        CUDA_CHECK(cudaEventSynchronize(ev_search_));
    }
    if (analyse) { /* results to the caller; this picture is the lane's next search reference */
        CUDA_CHECK(cudaStreamSynchronize(st));
        ktimes.collect(0);
        for (int k = 0; k < n; k++) {
            const int li = lane_ids[k];
            EncLane &l = lanes_[(size_t) li];
            LongAnalysis *out = plan[k].out;
            if (out) {
                out->luma_sum = inter_ ? h_misc[li].luma_sum : 0;
                out->nintra = l.has_ref ? h_misc[li].nintra : 0;
                if (l.has_ref && out->mvs) {
                    memcpy(out->mvs, h_mv0_ + (size_t) li * g.nblk, sizeof(DevMV) * (size_t) g.nblk);
                }
            }
            l.have_ref = 1;
            l.cur ^= 1;
            if (nbufs) {
                nbufs[k] = 0;
            }
        }
        stats.pictures += (unsigned) n;
        return;
    }

    /* ---- phase 2: host decisions + packet heads --------------------------------------------------- */
    const double t_host0 = host_now_ms();
    int n_p = 0, n_ref = 0;
    const std::function<void(int)> lane_head = [&](int k) {
        const int li = lane_ids[k];
        EncLane &l = lanes_[(size_t) li];
        if (code) { /* decided by the serial pass of dsvb_encode_long */
            l.quant = plan[k].quant;
            l.head_bytes = plan[k].head_bytes;
            memcpy(l.h_head, plan[k].head, plan[k].head_bytes);
            memcpy(h_stab_ + (size_t) li * g.nblk, plan[k].stable, (size_t) g.nblk);
            return;
        }
        DSV_ENCODER *enc = l.enc;
        const DevFrame *top = inter_ ? &l.pyr[l.cur][levels_ - 1] : nullptr;
        decide_and_head(enc, g, inter_, top ? top->w[0] * top->h[0] : 1, h_misc[li].luma_sum, h_misc[li].nintra,
                        h_mv0_ + (size_t) li * g.nblk, l.fnum, l.is_ref, &l.has_ref, &l.forced_intra, &l.quant, l.h_head, &l.head_bytes);
        memcpy(h_stab_ + (size_t) li * g.nblk, enc->stable_blocks, (size_t) g.nblk);
    };
    if (pool_) {
        pool_->run(n, lane_head);
    } else {
        for (int k = 0; k < n; k++) {
            lane_head(k);
        }
    }
    for (int k = 0; k < n; k++) {
        const EncLane &l = lanes_[(size_t) lane_ids[k]];
        n_p += l.has_ref;
        n_ref += l.is_ref;
    }
    stats.host_ms += host_now_ms() - t_host0;

    /* ---- phase 3: residual, transform, entropy coding, closed-loop reconstruction ------------------ */
    SbtJob *d_sj;
    HzJob *d_hj;
    HzFrame *d_hf = d_frames_;
    PlaneRef *d_ext = nullptr;
    SbtJob *sj = arena_.push_n<SbtJob>((size_t) 3 * n, &d_sj);
    HzJob *hj = arena_.push_n<HzJob>((size_t) 3 * n, &d_hj);
    PlaneRef *ext = n_ref > 0 ? arena_.push_n<PlaneRef>((size_t) 3 * n_ref, &d_ext) : nullptr;
    int qi = 0;
    ZeroItem *d_zero;
    ZeroItem *zero = arena_.push_n<ZeroItem>((size_t) 2 * n + (sse_on ? 1 : 0) + (ssim_on ? 1 : 0), &d_zero);
    int n_zero = 0;
    size_t max_zero = 0;
    SseJob *d_sse_jobs = nullptr, *d_ssim_jobs = nullptr;
    SseJob *sse_jobs = sse_on ? arena_.push_n<SseJob>((size_t) 3 * n, &d_sse_jobs) : nullptr;
    SseJob *ssim_jobs = ssim_on ? arena_.push_n<SseJob>((size_t) 3 * n, &d_ssim_jobs) : nullptr;
    for (int k = 0; k < n; k++) {
        const int li = lane_ids[k];
        EncLane &l = lanes_[(size_t) li];
        const int isP = l.has_ref;
        const DevFrame &fwd_in = isP ? l.xf : (inter_ ? l.pad[l.cur] : l.xf);
        /* P pictures: the inverse transform adds the prediction on its way out and writes the reconstruction */
        const DevFrame &inv_out = inter_ ? l.recon[l.cur] : (report ? l.qrec : l.xf);
        /* the ingested source against the reconstruction */
        if (sse_on) {
            sse_fill_picture(&sse_jobs[3 * k], g, inter_ ? l.pad[l.cur] : l.xf, inv_out, d_sse_ + 3 * k);
        }
        if (ssim_on) {
            sse_fill_picture(&ssim_jobs[3 * k], g, inter_ ? l.pad[l.cur] : l.xf, inv_out, d_ssim_ + 3 * k);
        }
        /* tile flags (sbt.cuh): the forward transform ORs into zeroed bytes */
        zero[n_zero].p = l.tflags;
        zero[n_zero].bytes = ((size_t) g.total_tiles + 15) & ~(size_t) 15;
        max_zero = max_zero > zero[n_zero].bytes ? max_zero : zero[n_zero].bytes;
        n_zero++;
        if (l.pkt_dirty) {
            zero[n_zero].p = l.d_pkt;
            zero[n_zero].bytes = ((size_t) l.pkt_dirty + 64 + 15) & ~(size_t) 15;
            max_zero = max_zero > zero[n_zero].bytes ? max_zero : zero[n_zero].bytes;
            n_zero++;
        }
        for (int p = 0; p < 3; p++) {
            EncPlaneIO io;
            io.in = fwd_in.p[p];
            io.in_stride = fwd_in.stride[p];
            io.out = inv_out.p[p];
            io.out_stride = inv_out.stride[p];
            io.pred = l.pred.p[p];
            io.pred_stride = l.pred.stride[p];
            io.coef = l.coef + g.coef_off[p];
            io.llx = l.llx[p];
            io.dv = l.dv[p];
            io.tflags = l.tflags;
            io.hz_dense = l.hz_dense;
            io.stable = d_stab_ + (size_t) li * g.nblk;
            enc_fill_plane(&sj[3 * k + p], &hj[3 * k + p], g, p, k, isP, l.quant, io);
            if (l.is_ref) {
                ext[3 * qi + p] = plane_ref(l.recon[l.cur], p);
            }
        }
        enc_fill_frame(&h_frames_[k], l.d_pkt, (unsigned) l.pkt_cap, l.head_bytes, k);
        if (l.is_ref) {
            qi++;
        }
    }
    for (unsigned long long *sums : {sse_on ? d_sse_ : nullptr, ssim_on ? d_ssim_ : nullptr}) {
        if (sums) {
            zero[n_zero].p = sums;
            zero[n_zero].bytes = (sizeof(unsigned long long) * 3 * (size_t) n + 15) & ~(size_t) 15;
            max_zero = max_zero > zero[n_zero].bytes ? max_zero : zero[n_zero].bytes;
            n_zero++;
        }
    }
    const SbtDims sdims = sbt_assign_tiles(sj, 3 * n);
    {
        CopyItem up[3] = {{nullptr, nullptr, 0}, {d_stab_, h_stab_, (size_t) g.nblk * L_}, {d_hf, h_frames_, sizeof(HzFrame) * (size_t) n}};
        arena_.take_upload(&up[0]);
        copyn_launch(up, 3, st);
    }
    zero_launch(d_zero, n_zero, max_zero, st);
    sbt_fwd_launch(d_sj, sdims, g.lo_smem, st, timed ? ev_[0] : nullptr, timed ? ev_[1] : nullptr);
    hzcc_enc_launch(d_hj, 3 * n, d_chunks_, n * g.total_chunks, d_hf, n, st, g.total_chunks, g.chunks[0], g.chunks[1], n_p < n);
    stats.kernel_launches += 6;
    copy1_launch(h_frames_, d_hf, sizeof(HzFrame) * (size_t) n, st);
    CUDA_CHECK(cudaEventRecord(ev_sizes_, st));
    /* the reports also need the reconstruction of pictures that are not references (intra-only engines) */
    const int n_inv = report ? n : n_ref;
    if (n_inv) {
        /* closed loop: reconstruct exactly what the decoder will (dsv_encoder.c:525,662-674) */
        sbt_inv_launch(d_sj, sdims, g.lo_smem, st, timed ? ev_[2] : nullptr, timed ? ev_[3] : nullptr);
        stats.kernel_launches += 3;
    }
    if (n_ref) {
        extend_launch(d_ext, 3 * n_ref, g.w, g.h, st);
        stats.kernel_launches += 1;
    }
    if (sse_on) {
        sse_launch(d_sse_jobs, 3 * n, g.h, st);
        stats.kernel_launches += 1;
    }
    if (ssim_on) {
        ssim_launch(d_ssim_jobs, 3 * n, g.w, g.h, st);
        stats.kernel_launches += 1;
    }
    CUDA_CHECK(cudaEventSynchronize(ev_sizes_)); /* packet sizes are known; reconstruction keeps running */
    CopyItem *pk = reinterpret_cast<CopyItem *>(h_pk_); /* mapped pinned: read by the copy kernel in place */
    int n_pk = 0;
    size_t max_pk = 0;

    for (int k = 0; k < n; k++) {
        EncLane &l = lanes_[(size_t) lane_ids[k]];
        DSV_ENCODER *enc = l.enc;
        const unsigned total = h_frames_[k].total_bytes;
        DSV_BUF outbuf;
        int nb = 0;
        if (h_frames_[k].overflow) { /* cannot happen for 8-bit input (see enc_packet_cap); never trust the size if it does */
            DSV_ERROR(("coded picture does not fit the packet buffer (%u bytes): picture dropped", (unsigned) l.pkt_cap));
            l.pkt_dirty = (unsigned) l.pkt_cap - 64;
            nbufs[k] = 0;
            if (sinks) {
                sinks[k].overflow = 1;
            }
            continue;
        }
        if (sinks) { /* caller-provided stream memory: metadata packet, then the picture, back to back */
            PktSink &sk = sinks[k];
            if (l.gop_start) {
                DSV_BUF meta;
                make_metadata_packet(enc, &meta);
                if (sk.room >= meta.len) {
                    memcpy(sk.at, meta.data, meta.len);
                    bufs[k][nb].data = sk.at;
                    bufs[k][nb].len = meta.len;
                    sk.at += meta.len;
                    sk.room -= meta.len;
                } else {
                    sk.overflow = 1;
                    bufs[k][nb].data = nullptr;
                    bufs[k][nb].len = 0;
                }
                nb++;
                dsv_buf_free(&meta);
            }
            if (sk.room >= total && !sk.overflow) {
                outbuf.data = sk.at;
                outbuf.len = total;
                sk.at += total;
                sk.room -= total;
            } else {
                sk.overflow = 1;
                outbuf.data = nullptr;
                outbuf.len = 0;
            }
        } else {
            dsv_mk_buf(&outbuf, (int) total + 8);
            outbuf.len = total;
            if (l.gop_start) {
                make_metadata_packet(enc, &bufs[k][nb++]);
            }
        }
        if (outbuf.data) {
            memcpy(outbuf.data, l.h_head, l.head_bytes);
            if (sinks && sinks[k].mapped) {
                pk[n_pk].dst = outbuf.data + l.head_bytes;
                pk[n_pk].src = l.d_pkt + l.head_bytes;
                pk[n_pk].bytes = total - l.head_bytes;
                max_pk = max_pk > pk[n_pk].bytes ? max_pk : pk[n_pk].bytes;
                n_pk++;
            } else {
                CUDA_CHECK(cudaMemcpyAsync(outbuf.data + l.head_bytes, l.d_pkt + l.head_bytes, total - l.head_bytes, cudaMemcpyDeviceToHost, st));
            }
            stats.d2h_bytes += total - l.head_bytes;
        }
        l.pkt_dirty = total;
        bufs[k][nb++] = outbuf;
        nbufs[k] = nb;
    }
    for (int r = 0; r < 2; r++) { /* the reports' sums leave with the packets */
        if (r == 0 ? sse_on : ssim_on) {
            pk[n_pk].dst = r == 0 ? h_sse_ : h_ssim_;
            pk[n_pk].src = r == 0 ? d_sse_ : d_ssim_;
            pk[n_pk].bytes = sizeof(unsigned long long) * 3 * (size_t) n;
            max_pk = max_pk > pk[n_pk].bytes ? max_pk : pk[n_pk].bytes;
            n_pk++;
        }
    }
    copy_launch(pk, n_pk, max_pk, st);
    CUDA_CHECK(cudaStreamSynchronize(st));
    ktimes.collect(0);
    stats.pictures += (unsigned) n;
    if (report) {
        pic_info.assign(sse_on ? (size_t) n : 0, DSVB_PICINFO());
        pic_ssim.assign(ssim_on ? (size_t) n : 0, DSVB_PICSSIM());
        pic_info_ok.assign((size_t) n, 0);
        for (int k = 0; k < n; k++) {
            const EncLane &l = lanes_[(size_t) lane_ids[k]];
            if (h_frames_[k].overflow) {
                continue;
            }
            pic_info_ok[(size_t) k] = 1;
            for (int p = 0; ssim_on && p < 3; p++) {
                DSVB_PICSSIM &s = pic_ssim[(size_t) k];
                s.windows[p] = ssim_windows(g.pw[p], g.ph[p]);
                s.ssim[p] = s.windows[p] ? (double) (int64_t) h_ssim_[3 * k + p] / 4294967296.0 / (double) s.windows[p] : NAN;
            }
            if (!sse_on) {
                continue;
            }
            DSVB_PICINFO &r = pic_info[(size_t) k];
            for (int p = 0; p < 3; p++) {
                r.sse[p] = h_sse_[3 * k + p];
                r.samples[p] = (int64_t) g.pw[p] * g.ph[p];
            }
            r.fnum = (int64_t) l.fnum;
            r.is_p = l.has_ref;
            r.forced_intra = plan ? plan[k].forced_intra : (inter_ && !l.has_ref && !l.gop_start);
            r.quant = l.quant;
            r.bytes = (int32_t) h_frames_[k].total_bytes;
        }
    }
    if (timed) {
        float ms = 0;
        CUDA_CHECK(cudaEventElapsedTime(&ms, ev_[0], ev_[1]));
        stats.sbt_fwd_ms += ms;
        stats.sbt_fwd_launches++;
        unsigned long long bytes = 0;
        for (int p = 0; p < 3; p++) {
            bytes += (unsigned long long) g.cw[p] * g.ph[p] + 4ull * g.cw[p] * g.ch[p];
        }
        stats.sbt_fwd_bytes += bytes * (unsigned) n;
        if (n_inv) {
            CUDA_CHECK(cudaEventElapsedTime(&ms, ev_[2], ev_[3]));
            stats.sbt_inv_ms += ms;
            stats.sbt_inv_launches++;
            /* P pictures also read the prediction (one more byte per sample) on the way out */
            stats.sbt_inv_bytes += bytes * (unsigned) n + (unsigned long long) g.frame_bytes * (unsigned) n_p;
        }
        if (n_search) {
            CUDA_CHECK(cudaEventElapsedTime(&ms, ev_[5], ev_[6]));
            stats.bmc_ms += ms;
            stats.bmc_launches++;
            stats.bmc_bytes += 4ull * g.frame_bytes * (unsigned) n_search;
        }
    }
    for (int k = 0; k < n; k++) {
        EncLane &l = lanes_[(size_t) lane_ids[k]];
        DSV_ENCODER *enc = l.enc;
        if (l.is_ref) {
            l.have_ref = 1;
            l.cur ^= 1;
        }
        if (plan) {
            continue; /* links and the serial state belong to the gather / the serial pass */
        }
        if (l.has_ref) {
            enc->refresh_ctr++;
        }
        if (nbufs[k] == 0) {
            continue; /* picture dropped (packet overflow) */
        }
        DSV_BUF *pic = &bufs[k][nbufs[k] - 1];
        if (pic->data) {
            rate_control_update(enc, l.has_ref, pic->len);
            set_links(enc, pic, 0);
        }
    }
}

} // namespace dsv

/* ---- public API ------------------------------------------------------------------------------ */

/* DSV_ENCODER.ref (the reference's "used internally" slot) holds the one-lane engine */
static EncEngine *enc_engine(DSV_ENCODER *enc) { return reinterpret_cast<EncEngine *>(enc->ref); }

extern "C" void dsv_enc_init(DSV_ENCODER *enc) /* defaults: dsv_encoder.c:696-722 */
{
    memset(enc, 0, sizeof(*enc));
    enc->prev_gop = (DSV_FNUM) -1;
    enc->quality = DSV_QUALITY_PERCENT(85);
    enc->gop = 24;
    enc->pyramid_levels = 0;
    enc->rc_mode = DSV_RATE_CONTROL_CRF;
    enc->bitrate = INT_MAX;
    enc->max_q_step = DSV_MAX_QUALITY / 200;
    enc->min_quality = DSV_QUALITY_PERCENT(1);
    enc->max_quality = DSV_QUALITY_PERCENT(95);
    enc->min_I_frame_quality = DSV_QUALITY_PERCENT(5);
    enc->rc_high_motion_nudge = 1;
    enc->intra_pct_thresh = 50;
    enc->stable_refresh = 14;
    enc->scene_change_delta = 4;
    enc->do_scd = 1;
}

extern "C" void dsv_enc_start(DSV_ENCODER *enc) /* dsv_encoder.c:724-734 */
{
    enc->quality = iclamp(enc->quality, 0, DSV_MAX_QUALITY);
    if (enc->rc_mode != DSV_RATE_CONTROL_CRF) {
        enc->rc_quant = (unsigned) enc->quality;
        enc->avg_P_frame_q = enc->quality * 4 / 5;
    }
    enc->force_metadata = 1;
}

extern "C" void dsv_enc_free(DSV_ENCODER *enc)
{
    delete enc_engine(enc);
    enc->ref = NULL;
    if (enc->stability) {
        dsv_free(enc->stability);
        enc->stability = NULL;
    }
    if (enc->stable_blocks) {
        dsv_free(enc->stable_blocks);
        enc->stable_blocks = NULL;
    }
}

extern "C" void dsv_enc_set_metadata(DSV_ENCODER *enc, DSV_META *md) { enc->vidmeta = *md; }
extern "C" void dsv_enc_force_metadata(DSV_ENCODER *enc) { enc->force_metadata = 1; }

extern "C" void dsv_enc_end_of_stream(DSV_ENCODER *enc, DSV_BUF *bufs) /* dsv_encoder.c:765-778 */
{
    dsv_mk_buf(&bufs[0], DSV_PACKET_HDR_SIZE);
    BitWriter bw(bufs[0].data);
    put_packet_hdr(bw, DSV_PT_EOS);
    set_links(enc, &bufs[0], 1);
}

/* block grid, stability arrays and pyramid depth (dsv_encoder.c:588-613): fixed for the life of the encoder */
void dsv::enc_prepare_state(DSV_ENCODER *enc)
{
    const int w = enc->vidmeta.width, h = enc->vidmeta.height;
    const int blk_w = iclamp(size4dim(w) & ~7, DSV_MIN_BLOCK_SIZE, DSV_MAX_BLOCK_SIZE);
    const int blk_h = iclamp(size4dim(h) & ~7, DSV_MIN_BLOCK_SIZE, DSV_MAX_BLOCK_SIZE);
    const int nbh = ceil_div(w, blk_w), nbv = ceil_div(h, blk_h);
    if (enc->stability == NULL) {
        enc->stability = (decltype(enc->stability)) dsv_alloc((int) sizeof(*enc->stability) * nbh * nbv);
        enc->stable_blocks = (unsigned char *) dsv_alloc(nbh * nbv);
    }
    if (enc->pyramid_levels == 0) {
        int lvls = lb2((unsigned) imin(w, h));
        int maxdim = imax(nbh, nbv);
        while ((1 << lvls) > maxdim) {
            lvls--;
        }
        enc->pyramid_levels = iclamp(lvls, 3, DSV_MAX_PYRAMID_LEVELS);
    }
}

extern "C" int dsv_enc(DSV_ENCODER *enc, DSV_FRAME *frame, DSV_BUF *bufs)
{
    DSV_API_BEGIN
    if (bufs == NULL) {
        DSV_ERROR(("null buffer list passed to encoder!"));
        return 0;
    }
    enc_prepare_state(enc);
    if (enc->ref == NULL) { /* created on the first call, when metadata, gop and pyramid settings are final */
        EncEngine *e = new EncEngine(enc->vidmeta, enc->gop, enc->pyramid_levels, 1);
        e->bind(0, enc);
        enc->ref = reinterpret_cast<DSV_ENCDATA *>(e);
    }
    EncEngine *e = enc_engine(enc);
    PicRef src;
    for (int p = 0; p < 3; p++) {
        src.plane[p] = frame->planes[p].data;
        src.stride[p] = frame->planes[p].stride;
    }
    src.on_device = 0;
    const int lane = 0;
    DSV_BUF out[1][2];
    int nb = 0;
    e->step(1, &lane, &src, out, &nb);
    dsv_frame_ref_dec(frame); /* the encoder owns the reference it was given (dsv_encoder.c:38-40,801) */
    for (int i = 0; i < nb; i++) {
        bufs[i] = out[0][i];
    }
    return nb;
    DSV_API_END(0)
}
