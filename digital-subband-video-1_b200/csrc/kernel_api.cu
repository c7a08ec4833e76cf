/*
 * kernel_api.cu -- dsvk_*: kernel-level C ABI with HOST buffers (declared in include/dsv1_b200_kernels.h).
 *
 * One entry point per hot-path subsystem, with the same flat signatures as the checker libraries
 * (oracle/ref_harness.c, oracle/dsv1_port.c) so the parity tests call all three alike.  Every call
 * copies its inputs to the GPU, runs the CUDA kernels and copies the result back: there is no host
 * implementation behind these symbols.
 */
#include "common.cuh"
#include "sbt.cuh"
#include "hzcc.cuh"
#include "hzcc_dec.cuh"
#include "frame.cuh"
#include "motion.cuh"
#include "dsv1_b200.h"
#include "dsv1_b200_kernels.h"
#include "host/engine.h"

#include <vector>

using namespace dsv;

namespace {

struct DevBuf {
    void *p = nullptr;
    explicit DevBuf(size_t n) { CUDA_CHECK(cudaMalloc(&p, n ? n : 1)); }
    ~DevBuf() { cudaFree(p); }
    template <typename T> T *as() { return reinterpret_cast<T *>(p); }
};

/* device plane in the reference's bordered layout: returns pointer to sample (0,0) */
struct DevPlane {
    DevBuf buf;
    int stride, rows;
    uint8_t *origin;
    DevPlane(int w, int h)
        : buf((size_t) frame_stride(w) * (h + 2 * DSV_BORDER) + 256), stride(frame_stride(w)), rows(h + 2 * DSV_BORDER)
    {
        CUDA_CHECK(cudaMemset(buf.p, 0, (size_t) stride * rows + 256));
        origin = buf.as<uint8_t>() + (size_t) stride * DSV_BORDER + DSV_BORDER;
    }
};

} // namespace

extern "C" int dsvk_fwd_sbt(const uint8_t *pix, int stride, int pw, int ph, int cw, int ch, int isP, int32_t *coef_out)
{
    DSV_API_BEGIN
    if ((cw & 1) || (ch & 1) || cw < 16 || ch < 16) {
        return -1;
    }
    DevPlane dp(cw, ph);
    CUDA_CHECK(cudaMemcpy2D(dp.origin, dp.stride, pix, stride, cw, ph, cudaMemcpyHostToDevice));
    DevBuf coef((size_t) cw * ch * 4), llx(sbt_llx_elems(cw, ch) * 4), dv(sbt_dv_elems(cw, ch) * 4), jobs(sizeof(SbtJob));
    CUDA_CHECK(cudaMemset(coef.p, 0, (size_t) cw * ch * 4));
    SbtJob j;
    memset(&j, 0, sizeof(j));
    sbt_fill_geometry(&j, pw, ph, cw, ch, isP, 0);
    j.pix = dp.origin;
    j.pstride = dp.stride;
    j.coef = coef.as<int32_t>();
    j.llx = llx.as<int32_t>();
    j.dv = dv.as<int32_t>();
    j.do_quant = 0;
    const SbtDims dims = sbt_assign_tiles(&j, 1);
    CUDA_CHECK(cudaMemcpy(jobs.p, &j, sizeof(j), cudaMemcpyHostToDevice));
    sbt_fwd_launch(jobs.as<SbtJob>(), dims, sbt_lo_smem_bytes(cw, ch), 0);
    CUDA_CHECK(cudaDeviceSynchronize());
    CUDA_CHECK(cudaMemcpy(coef_out, coef.p, (size_t) cw * ch * 4, cudaMemcpyDeviceToHost));
    return 0;
    DSV_API_END(-100)
}

extern "C" int dsvk_inv_sbt(int32_t *coef_io, int cw, int ch, int q, int isP, int c, uint8_t *pix_out, int stride, int pw, int ph)
{
    DSV_API_BEGIN
    if ((cw & 1) || (ch & 1) || cw < 16 || ch < 16) {
        return -1;
    }
    DevPlane dp(cw, ph);
    DevBuf coef((size_t) cw * ch * 4), llx(sbt_llx_elems(cw, ch) * 4), jobs(sizeof(SbtJob));
    CUDA_CHECK(cudaMemcpy(coef.p, coef_io, (size_t) cw * ch * 4, cudaMemcpyHostToDevice));
    SbtJob j;
    memset(&j, 0, sizeof(j));
    sbt_fill_geometry(&j, pw, ph, cw, ch, isP, c);
    sbt_fill_quant(&j, q, isP, c, 1, 1);
    j.pix = dp.origin;
    j.pstride = dp.stride;
    j.opix = dp.origin;
    j.ostride = dp.stride;
    j.coef = coef.as<int32_t>();
    j.llx = llx.as<int32_t>();
    const SbtDims dims = sbt_assign_tiles(&j, 1);
    CUDA_CHECK(cudaMemcpy(jobs.p, &j, sizeof(j), cudaMemcpyHostToDevice));
    sbt_inv_launch(jobs.as<SbtJob>(), dims, sbt_lo_smem_bytes(cw, ch), 0);
    CUDA_CHECK(cudaDeviceSynchronize());
    CUDA_CHECK(cudaMemcpy2D(pix_out, stride, dp.origin, dp.stride, pw, ph, cudaMemcpyDeviceToHost));
    return 0;
    DSV_API_END(-100)
}

/* forward transform with the fused quantiser, exactly as the encoder runs it (do_quant = 1) */
extern "C" int dsvk_fwd_sbt_q(const uint8_t *pix, int stride, int pw, int ph, int cw, int ch, int isP, int c, int q,
                              const uint8_t *stable, int nbh, int nbv, int32_t *coef_out, int32_t *dv_out)
{
    DSV_API_BEGIN
    if ((cw & 1) || (ch & 1) || cw < 16 || ch < 16) {
        return -1;
    }
    DevPlane dp(cw, ph);
    CUDA_CHECK(cudaMemcpy2D(dp.origin, dp.stride, pix, stride, cw, ph, cudaMemcpyHostToDevice));
    DevBuf coef((size_t) cw * ch * 4), llx(sbt_llx_elems(cw, ch) * 4), dv(sbt_dv_elems(cw, ch) * 4), jobs(sizeof(SbtJob));
    DevBuf stab((size_t) nbh * nbv);
    CUDA_CHECK(cudaMemset(coef.p, 0, (size_t) cw * ch * 4));
    CUDA_CHECK(cudaMemset(dv.p, 0, sbt_dv_elems(cw, ch) * 4));
    CUDA_CHECK(cudaMemcpy(stab.p, stable, (size_t) nbh * nbv, cudaMemcpyHostToDevice));
    SbtJob j;
    memset(&j, 0, sizeof(j));
    sbt_fill_geometry(&j, pw, ph, cw, ch, isP, c);
    sbt_fill_quant(&j, q, isP, c, nbh, nbv);
    j.pix = dp.origin;
    j.pstride = dp.stride;
    j.coef = coef.as<int32_t>();
    j.llx = llx.as<int32_t>();
    j.dv = dv.as<int32_t>();
    j.stable = stab.as<uint8_t>();
    j.do_quant = 1;
    const SbtDims dims = sbt_assign_tiles(&j, 1);
    CUDA_CHECK(cudaMemcpy(jobs.p, &j, sizeof(j), cudaMemcpyHostToDevice));
    sbt_fwd_launch(jobs.as<SbtJob>(), dims, sbt_lo_smem_bytes(cw, ch), 0);
    CUDA_CHECK(cudaDeviceSynchronize());
    CUDA_CHECK(cudaMemcpy(coef_out, coef.p, (size_t) cw * ch * 4, cudaMemcpyDeviceToHost));
    if (dv_out) {
        CUDA_CHECK(cudaMemcpy(dv_out, dv.p, (size_t) j.dg.total * 4, cudaMemcpyDeviceToHost));
    }
    return j.dg.total;
    DSV_API_END(-100)
}

/* dsv_encode_plane semantics (hzcc.c:449-476): raw coefficients in, plane bytes out, coef <- dequantised */
extern "C" int dsvk_encode_plane(int32_t *coef_io, int cw, int ch, int q, int isP, int c, const uint8_t *stable,
                                 int nbh, int nbv, uint8_t *out, int out_cap)
{
    DSV_API_BEGIN
    if ((cw & 1) || (ch & 1) || cw < 16 || ch < 16) {
        return -1;
    }
    HzJob j;
    memset(&j, 0, sizeof(j));
    hz_fill_job(&j, cw, ch, q, isP, c, nbh, nbv);
    const size_t cap = (size_t) cw * ch * 8 + 256;
    DevBuf coef((size_t) cw * ch * 4), dv(sbt_dv_elems(cw, ch) * 4), stab((size_t) nbh * nbv), pkt(cap);
    DevBuf jobs(sizeof(HzJob)), chunks(sizeof(HzChunk) * j.nchunks), frames(sizeof(HzFrame));
    CUDA_CHECK(cudaMemcpy(coef.p, coef_io, (size_t) cw * ch * 4, cudaMemcpyHostToDevice));
    CUDA_CHECK(cudaMemcpy(stab.p, stable, (size_t) nbh * nbv, cudaMemcpyHostToDevice));
    CUDA_CHECK(cudaMemset(dv.p, 0, sbt_dv_elems(cw, ch) * 4));
    CUDA_CHECK(cudaMemset(pkt.p, 0, cap));
    j.coef = coef.as<int32_t>();
    j.dv = dv.as<int32_t>();
    j.stable = stab.as<uint8_t>();
    j.chunk_base = 0;
    j.frame = 0;
    HzFrame f;
    memset(&f, 0, sizeof(f));
    f.pkt = pkt.as<uint8_t>();
    f.start_byte = 0;
    f.cap = (unsigned) cap;
    f.nplanes = 1;
    CUDA_CHECK(cudaMemcpy(jobs.p, &j, sizeof(j), cudaMemcpyHostToDevice));
    CUDA_CHECK(cudaMemcpy(frames.p, &f, sizeof(f), cudaMemcpyHostToDevice));
    hzcc_quant_launch(jobs.as<HzJob>(), 1, cw * ch, 0);
    hzcc_enc_launch(jobs.as<HzJob>(), 1, chunks.as<HzChunk>(), j.nchunks, frames.as<HzFrame>(), 1, 0);
    CUDA_CHECK(cudaDeviceSynchronize());
    CUDA_CHECK(cudaMemcpy(&f, frames.p, sizeof(f), cudaMemcpyDeviceToHost));
    if (f.overflow || (int) f.total_bytes > out_cap) {
        return -2;
    }
    CUDA_CHECK(cudaMemcpy(out, pkt.p, f.total_bytes, cudaMemcpyDeviceToHost));
    CUDA_CHECK(cudaMemcpy(coef_io, coef.p, (size_t) cw * ch * 4, cudaMemcpyDeviceToHost));
    return (int) f.total_bytes;
    DSV_API_END(-100)
}

/* dsv_decode_plane semantics (hzcc.c:478-496): `in` points just after the 32-bit plen field */
extern "C" int dsvk_decode_plane(const uint8_t *in, int plen, int cw, int ch, int q, int isP, int c,
                                 const uint8_t *stable, int nbh, int nbv, int32_t *coef_out)
{
    DSV_API_BEGIN
    if ((cw & 1) || (ch & 1) || cw < 16 || ch < 16 || plen <= 0) {
        return -1;
    }
    HzJob j;
    memset(&j, 0, sizeof(j));
    hz_fill_job(&j, cw, ch, q, isP, c, nbh, nbv);
    DevBuf coef((size_t) cw * ch * 4), stab((size_t) nbh * nbv), body((size_t) plen + 64);
    CUDA_CHECK(cudaMemset(coef.p, 0, (size_t) cw * ch * 4));
    CUDA_CHECK(cudaMemset(body.p, 0, (size_t) plen + 64));
    CUDA_CHECK(cudaMemcpy(body.p, in, (size_t) plen, cudaMemcpyHostToDevice));
    CUDA_CHECK(cudaMemcpy(stab.p, stable, (size_t) nbh * nbv, cudaMemcpyHostToDevice));
    j.coef = coef.as<int32_t>();
    j.stable = stab.as<uint8_t>();
    HzPlaneData pd;
    hzdec_parse_head(in, (unsigned) plen, (unsigned) plen, &pd);
    pd.body = body.as<uint8_t>();
    HzDecPlan pl;
    hzdec_plan(&pl, cw, ch);
    HzDecPlaneBufs bufs;
    hzdec_plane_alloc(&bufs, pl);
    HzDecDims dims;
    std::vector<uint8_t> slot(hzdec_job_size());
    hzdec_fill_job(slot.data(), j, pd, bufs, &dims);
    DevBuf djob(hzdec_job_size());
    CUDA_CHECK(cudaMemcpy(djob.p, slot.data(), hzdec_job_size(), cudaMemcpyHostToDevice));
    hzdec_launch_jobs(djob.p, dims, 0);
    CUDA_CHECK(cudaDeviceSynchronize());
    CUDA_CHECK(cudaMemcpy(coef_out, coef.p, (size_t) cw * ch * 4, cudaMemcpyDeviceToHost));
    hzdec_plane_free(&bufs);
    return 0;
    DSV_API_END(-100)
}

/* ---- motion: pyramid, HME, BMC ------------------------------------------------------------------ */

namespace {

/* packed planar YUV (host) -> bordered device frame, borders replicated (dsv_frame_copy + extend) */
void upload_frame(DevFrame *f, const uint8_t *yuv, int w, int h, int subsamp)
{
    devframe_alloc(f, w, h, subsamp);
    const uint8_t *s = yuv;
    for (int c = 0; c < 3; c++) {
        CUDA_CHECK(cudaMemcpy2D(f->p[c], f->stride[c], s, f->w[c], f->w[c], f->h[c], cudaMemcpyHostToDevice));
        s += (size_t) f->w[c] * f->h[c];
    }
    frame_extend_launch(*f, 3, 0);
}

void download_frame(const DevFrame &f, uint8_t *yuv)
{
    uint8_t *o = yuv;
    for (int c = 0; c < 3; c++) {
        CUDA_CHECK(cudaMemcpy2D(o, f.w[c], f.p[c], f.stride[c], f.w[c], f.h[c], cudaMemcpyDeviceToHost));
        o += (size_t) f.w[c] * f.h[c];
    }
}

MotionGeom motion_geom(int w, int h, int subsamp, int blk_w, int blk_h, int levels)
{
    MotionGeom g;
    g.w = w;
    g.h = h;
    g.hs = (subsamp >> 2) & 3;
    g.vs = subsamp & 3;
    g.blk_w = blk_w;
    g.blk_h = blk_h;
    g.nbh = ceil_div(w, blk_w);
    g.nbv = ceil_div(h, blk_h);
    g.levels = levels;
    return g;
}

} // namespace

extern "C" int dsvk_pyramid(const uint8_t *yuv, int w, int h, int subsamp, int levels, uint8_t *out, int *out_w, int *out_h)
{
    DSV_API_BEGIN
    if (levels < 1 || levels > 5) {
        return -1;
    }
    DevFrame f[6];
    upload_frame(&f[0], yuv, w, h, subsamp);
    for (int l = 0; l < levels; l++) {
        devframe_alloc(&f[l + 1], ceil_shift(w, l + 1), ceil_shift(h, l + 1), subsamp);
        frame_down2_luma_launch(f[l], f[l + 1], 0);
    }
    CUDA_CHECK(cudaDeviceSynchronize());
    for (int l = 1; l <= levels; l++) {
        CUDA_CHECK(cudaMemcpy2D(out, f[l].w[0], f[l].p[0], f[l].stride[0], f[l].w[0], f[l].h[0], cudaMemcpyDeviceToHost));
        out += (size_t) f[l].w[0] * f[l].h[0];
        out_w[l - 1] = f[l].w[0];
        out_h[l - 1] = f[l].h[0];
    }
    for (int l = 0; l <= levels; l++) {
        devframe_free(&f[l]);
    }
    return 0;
    DSV_API_END(-100)
}

extern "C" int dsvk_hme(const uint8_t *src_yuv, const uint8_t *ref_yuv, int w, int h, int subsamp, int blk_w, int blk_h,
                        int levels, void *mv_out)
{
    DSV_API_BEGIN
    if (levels < 0 || levels > 5) {
        return -1;
    }
    const MotionGeom g = motion_geom(w, h, subsamp, blk_w, blk_h, levels);
    const int nblk = g.nbh * g.nbv;
    DevFrame sf[6], rf[6];
    upload_frame(&sf[0], src_yuv, w, h, subsamp);
    upload_frame(&rf[0], ref_yuv, w, h, subsamp);
    for (int l = 0; l < levels; l++) {
        devframe_alloc(&sf[l + 1], ceil_shift(w, l + 1), ceil_shift(h, l + 1), subsamp);
        devframe_alloc(&rf[l + 1], ceil_shift(w, l + 1), ceil_shift(h, l + 1), subsamp);
        frame_down2_luma_launch(sf[l], sf[l + 1], 0);
        frame_down2_luma_launch(rf[l], rf[l + 1], 0);
    }
    DevMV *mvf[6];
    for (int l = 0; l <= levels; l++) {
        CUDA_CHECK(cudaMalloc(&mvf[l], sizeof(DevMV) * (size_t) nblk));
        CUDA_CHECK(cudaMemset(mvf[l], 0, sizeof(DevMV) * (size_t) nblk));
    }
    DevBuf aux(sizeof(int2) * (size_t) nblk), cnt(sizeof(int)), dargs(sizeof(HmeArgs) * (size_t) (levels + 1));
    CUDA_CHECK(cudaMemset(cnt.p, 0, sizeof(int)));
    std::vector<HmeArgs> ha((size_t) levels + 1);
    for (int l = 0; l <= levels; l++) {
        hme_fill_args(&ha[(size_t) l], g, l, sf, rf, mvf, aux.as<int2>(), cnt.as<int>());
    }
    CUDA_CHECK(cudaMemcpy(dargs.p, ha.data(), sizeof(HmeArgs) * ha.size(), cudaMemcpyHostToDevice));
    hme_launch(dargs.as<HmeArgs>(), 1, g, 0);
    CUDA_CHECK(cudaDeviceSynchronize());
    int nintra = 0;
    CUDA_CHECK(cudaMemcpy(&nintra, cnt.p, sizeof(int), cudaMemcpyDeviceToHost));
    CUDA_CHECK(cudaMemcpy(mv_out, mvf[0], sizeof(DevMV) * (size_t) nblk, cudaMemcpyDeviceToHost));
    for (int l = 0; l <= levels; l++) {
        cudaFree(mvf[l]);
        devframe_free(&sf[l]);
        devframe_free(&rf[l]);
    }
    return nintra * 100 / nblk;
    DSV_API_END(-100)
}

/* a caller's host frame -> device frame, border included when the caller's frame has one (the search reads it) */
static void upload_host_frame(DevFrame *f, const DSV_FRAME *src)
{
    devframe_alloc(f, src->width, src->height, src->format);
    for (int c = 0; c < 3; c++) {
        const DSV_PLANE &pl = src->planes[c];
        if (src->border && pl.stride >= pl.w + 2 * DSV_BORDER) {
            const int rows = pl.h + 2 * DSV_BORDER, cols = pl.w + 2 * DSV_BORDER;
            CUDA_CHECK(cudaMemcpy2D(f->p[c] - (ptrdiff_t) DSV_BORDER * f->stride[c] - DSV_BORDER, (size_t) f->stride[c],
                                    pl.data - (ptrdiff_t) DSV_BORDER * pl.stride - DSV_BORDER, (size_t) pl.stride, (size_t) cols, (size_t) rows,
                                    cudaMemcpyHostToDevice));
        } else {
            CUDA_CHECK(cudaMemcpy2D(f->p[c], (size_t) f->stride[c], pl.data, (size_t) pl.stride, (size_t) pl.w, (size_t) pl.h, cudaMemcpyHostToDevice));
        }
    }
    if (!src->border) {
        frame_extend_launch(*f, 3, 0);
    }
}

/* drop-in for the reference's exported dsv_hme (dsv_encoder.h:122-132, hme.c:730-741) */
extern "C" int dsv_hme(DSV_HME *hme)
{
    DSV_API_BEGIN
    const DSV_PARAMS *pr = hme->params;
    const int levels = hme->levels;
    if (levels < 0 || levels > DSV_MAX_PYRAMID_LEVELS) {
        return 0;
    }
    const DSV_FRAME *top = hme->src[0];
    MotionGeom g = motion_geom(top->width, top->height, top->format, pr->blk_w, pr->blk_h, levels);
    g.nbh = pr->nblocks_h;
    g.nbv = pr->nblocks_v;
    const int nblk = g.nbh * g.nbv;
    DevFrame sf[DSV_MAX_PYRAMID_LEVELS + 1], rf[DSV_MAX_PYRAMID_LEVELS + 1];
    DevMV *mvf[DSV_MAX_PYRAMID_LEVELS + 1];
    for (int l = 0; l <= levels; l++) {
        upload_host_frame(&sf[l], hme->src[l]);
        upload_host_frame(&rf[l], hme->ref[l]);
        CUDA_CHECK(cudaMalloc(&mvf[l], sizeof(DevMV) * (size_t) nblk));
        CUDA_CHECK(cudaMemset(mvf[l], 0, sizeof(DevMV) * (size_t) nblk));
    }
    DevBuf aux(sizeof(int2) * (size_t) nblk), cnt(sizeof(int)), dargs(sizeof(HmeArgs) * (size_t) (levels + 1));
    CUDA_CHECK(cudaMemset(cnt.p, 0, sizeof(int)));
    std::vector<HmeArgs> ha((size_t) levels + 1);
    for (int l = 0; l <= levels; l++) {
        hme_fill_args(&ha[(size_t) l], g, l, sf, rf, mvf, aux.as<int2>(), cnt.as<int>());
    }
    CUDA_CHECK(cudaMemcpy(dargs.p, ha.data(), sizeof(HmeArgs) * ha.size(), cudaMemcpyHostToDevice));
    hme_launch(dargs.as<HmeArgs>(), 1, g, 0);
    CUDA_CHECK(cudaDeviceSynchronize());
    int nintra = 0;
    CUDA_CHECK(cudaMemcpy(&nintra, cnt.p, sizeof(int), cudaMemcpyDeviceToHost));
    static_assert(sizeof(DSV_MV) == sizeof(DevMV), "DevMV is the device twin of DSV_MV");
    for (int l = 0; l <= levels; l++) {
        hme->mvf[l] = (DSV_MV *) dsv_alloc((int) (sizeof(DSV_MV) * (size_t) nblk));
        CUDA_CHECK(cudaMemcpy(hme->mvf[l], mvf[l], sizeof(DevMV) * (size_t) nblk, cudaMemcpyDeviceToHost));
        cudaFree(mvf[l]);
        devframe_free(&sf[l]);
        devframe_free(&rf[l]);
    }
    return nintra * 100 / nblk;
    DSV_API_END(-100)
}

extern "C" int dsvk_sub_pred(const void *mvs, int w, int h, int subsamp, int blk_w, int blk_h, const uint8_t *inp_yuv,
                             const uint8_t *ref_yuv, uint8_t *pred_out, uint8_t *resid_out)
{
    DSV_API_BEGIN
    const MotionGeom g = motion_geom(w, h, subsamp, blk_w, blk_h, 0);
    DevFrame inp, ref, pred;
    upload_frame(&inp, inp_yuv, w, h, subsamp);
    upload_frame(&ref, ref_yuv, w, h, subsamp);
    devframe_alloc(&pred, w, h, subsamp);
    DevBuf mv(sizeof(DevMV) * (size_t) g.nbh * g.nbv);
    CUDA_CHECK(cudaMemcpy(mv.p, mvs, sizeof(DevMV) * (size_t) g.nbh * g.nbv, cudaMemcpyHostToDevice));
    BmcArgs ba;
    bmc_fill_args(&ba, g, mv.as<DevMV>(), ref, &pred, inp, inp, 1);
    DevBuf dargs(sizeof(BmcArgs));
    CUDA_CHECK(cudaMemcpy(dargs.p, &ba, sizeof(ba), cudaMemcpyHostToDevice));
    bmc_launch(dargs.as<BmcArgs>(), 1, g, 0);
    CUDA_CHECK(cudaDeviceSynchronize());
    download_frame(pred, pred_out);
    download_frame(inp, resid_out);
    devframe_free(&inp);
    devframe_free(&ref);
    devframe_free(&pred);
    return 0;
    DSV_API_END(-100)
}

extern "C" int dsvk_add_pred(const void *mvs, int w, int h, int subsamp, int blk_w, int blk_h, const uint8_t *resid_yuv,
                             const uint8_t *ref_yuv, uint8_t *out_yuv)
{
    DSV_API_BEGIN
    const MotionGeom g = motion_geom(w, h, subsamp, blk_w, blk_h, 0);
    DevFrame io, ref;
    upload_frame(&io, resid_yuv, w, h, subsamp);
    upload_frame(&ref, ref_yuv, w, h, subsamp);
    DevBuf mv(sizeof(DevMV) * (size_t) g.nbh * g.nbv);
    CUDA_CHECK(cudaMemcpy(mv.p, mvs, sizeof(DevMV) * (size_t) g.nbh * g.nbv, cudaMemcpyHostToDevice));
    BmcArgs ba;
    bmc_fill_args(&ba, g, mv.as<DevMV>(), ref, nullptr, io, io, 2);
    DevBuf dargs(sizeof(BmcArgs));
    CUDA_CHECK(cudaMemcpy(dargs.p, &ba, sizeof(ba), cudaMemcpyHostToDevice));
    bmc_launch(dargs.as<BmcArgs>(), 1, g, 0);
    CUDA_CHECK(cudaDeviceSynchronize());
    download_frame(io, out_yuv);
    devframe_free(&io);
    devframe_free(&ref);
    return 0;
    DSV_API_END(-100)
}

/* ---- batch entry points: the engines' own job filling and launch sequence (host/plane_jobs.cpp) ------------------- */
namespace {

template <typename T> T *dev_alloc(size_t n, bool zero = true)
{
    T *p = nullptr;
    CUDA_CHECK(cudaMalloc(&p, n * sizeof(T) + 16));
    if (zero) {
        CUDA_CHECK(cudaMemset(p, 0, n * sizeof(T) + 16));
    }
    return p;
}

void upload_packed(const DevFrame &f, const uint8_t *src)
{
    for (int c = 0; c < 3; c++) {
        CUDA_CHECK(cudaMemcpy2D(f.p[c], f.stride[c], src, f.w[c], f.w[c], f.h[c], cudaMemcpyHostToDevice));
        src += (size_t) f.w[c] * f.h[c];
    }
}

} // namespace

#define DSVK_PKT_GUARD 4096 /* bytes past the largest cap, where nothing may ever be written */

/* EncEngine's lanes, lane k = picture k: its phase 3 reads the picture from xf and the prediction from pred, and leaves
 * the reconstruction in recon[0] */
struct DsvkEnc {
    CodecGeom g;
    int max_pics;
    size_t pkt_bytes, dv_pitch;
    std::vector<EncLane> lanes;
    HzChunk *chunks = nullptr;
    HzFrame *frames = nullptr;
    SbtJob *d_sj = nullptr;
    HzJob *d_hj = nullptr;
    ZeroItem *d_zero = nullptr;
};

extern "C" void *dsvk_enc_create(int w, int h, int subsamp, int blk_w, int blk_h, int max_pics)
{
    DSV_API_BEGIN
    if (w < 16 || h < 16 || (w & 1) || (h & 1) || max_pics < 1) {
        return nullptr;
    }
    DsvkEnc *e = new DsvkEnc;
    plan_geometry(&e->g, w, h, subsamp);
    plan_blocks(&e->g, blk_w, blk_h);
    const CodecGeom &g = e->g;
    e->max_pics = max_pics;
    e->pkt_bytes = enc_packet_cap(g);
    e->dv_pitch = sbt_dv_elems(g.cw[0], g.ch[0]);
    e->lanes.resize((size_t) max_pics);
    for (auto &l : e->lanes) {
        enc_lane_alloc(l, g, true, 0, e->pkt_bytes + DSVK_PKT_GUARD);
    }
    e->chunks = dev_alloc<HzChunk>((size_t) max_pics * g.total_chunks, false);
    e->frames = dev_alloc<HzFrame>((size_t) max_pics);
    e->d_sj = dev_alloc<SbtJob>((size_t) 3 * max_pics);
    e->d_hj = dev_alloc<HzJob>((size_t) 3 * max_pics);
    e->d_zero = dev_alloc<ZeroItem>((size_t) 2 * max_pics);
    return e;
    DSV_API_END(nullptr)
}

extern "C" long dsvk_enc_pkt_bytes(void *handle) { return (long) static_cast<DsvkEnc *>(handle)->pkt_bytes; }

extern "C" void dsvk_enc_destroy(void *handle)
{
    DsvkEnc *e = static_cast<DsvkEnc *>(handle);
    if (!e) {
        return;
    }
    for (auto &l : e->lanes) {
        enc_lane_free(l);
    }
    cudaFree(e->chunks);
    cudaFree(e->frames);
    cudaFree(e->d_sj);
    cudaFree(e->d_hj);
    cudaFree(e->d_zero);
    delete e;
}

/* phase 3 of EncEngine::step (encoder.cpp) on n pictures, lane k = picture k */
extern "C" int dsvk_enc_run(void *handle, int n, const DSVK_PIC *pics, const uint8_t *in, const uint8_t *pred, uint8_t *pkt_out,
                            unsigned *info_out, int32_t *coef_out, int32_t *dv_out, uint8_t *tflags_out, uint8_t *recon_out)
{
    DSV_API_BEGIN
    DsvkEnc *e = static_cast<DsvkEnc *>(handle);
    const CodecGeom &g = e->g;
    if (n < 1 || n > e->max_pics) {
        return -1;
    }
    std::vector<SbtJob> sj((size_t) 3 * n);
    std::vector<HzJob> hj((size_t) 3 * n);
    std::vector<HzFrame> hf((size_t) n);
    std::vector<ZeroItem> zero;
    size_t max_zero = 0;
    int n_p = 0;
    for (int k = 0; k < n; k++) {
        EncLane &l = e->lanes[(size_t) k];
        const DSVK_PIC &pc = pics[k];
        if (pc.cap > e->pkt_bytes || pc.start_byte + 64 > pc.cap) {
            return -1;
        }
        upload_packed(l.xf, in + g.frame_bytes * k);
        if (pred && pc.isP) {
            upload_packed(l.pred, pred + g.frame_bytes * k);
        }
        /* as the engine: the forward transform ORs its tile flags into zeroed bytes; the packet's dirty prefix is cleared */
        zero.push_back({l.tflags, ((size_t) g.total_tiles + 15) & ~(size_t) 15});
        if (l.pkt_dirty) {
            zero.push_back({l.d_pkt, ((size_t) l.pkt_dirty + 64 + 15) & ~(size_t) 15});
        }
        n_p += pc.isP != 0;
    }
    for (const ZeroItem &z : zero) {
        max_zero = max_zero > z.bytes ? max_zero : z.bytes;
    }
    uint8_t *d_stab = dev_alloc<uint8_t>((size_t) g.nblk * n, false);
    for (int k = 0; k < n; k++) {
        CUDA_CHECK(cudaMemcpy(d_stab + (size_t) g.nblk * k, pics[k].stable, (size_t) g.nblk, cudaMemcpyHostToDevice));
        EncLane &l = e->lanes[(size_t) k];
        const int isP = pics[k].isP != 0;
        for (int p = 0; p < 3; p++) {
            EncPlaneIO io;
            io.in = l.xf.p[p];
            io.in_stride = l.xf.stride[p];
            io.out = l.recon[0].p[p];
            io.out_stride = l.recon[0].stride[p];
            io.pred = pred ? l.pred.p[p] : nullptr;
            io.pred_stride = l.pred.stride[p];
            io.coef = l.coef + g.coef_off[p];
            io.llx = l.llx[p];
            io.dv = l.dv[p];
            io.tflags = l.tflags;
            io.hz_dense = l.hz_dense;
            io.stable = d_stab + (size_t) g.nblk * k;
            enc_fill_plane(&sj[(size_t) 3 * k + p], &hj[(size_t) 3 * k + p], g, p, k, isP, pics[k].quant, io);
        }
        enc_fill_frame(&hf[(size_t) k], l.d_pkt, pics[k].cap, pics[k].start_byte, k);
    }
    const SbtDims sdims = sbt_assign_tiles(sj.data(), 3 * n);
    CUDA_CHECK(cudaMemcpy(e->d_sj, sj.data(), sizeof(SbtJob) * sj.size(), cudaMemcpyHostToDevice));
    CUDA_CHECK(cudaMemcpy(e->d_hj, hj.data(), sizeof(HzJob) * hj.size(), cudaMemcpyHostToDevice));
    CUDA_CHECK(cudaMemcpy(e->frames, hf.data(), sizeof(HzFrame) * hf.size(), cudaMemcpyHostToDevice));
    CUDA_CHECK(cudaMemcpy(e->d_zero, zero.data(), sizeof(ZeroItem) * zero.size(), cudaMemcpyHostToDevice));
    zero_launch(e->d_zero, (int) zero.size(), max_zero, 0);
    sbt_fwd_launch(e->d_sj, sdims, g.lo_smem, 0);
    hzcc_enc_launch(e->d_hj, 3 * n, e->chunks, n * g.total_chunks, e->frames, n, 0, g.total_chunks, g.chunks[0], g.chunks[1], n_p < n);
    sbt_inv_launch(e->d_sj, sdims, g.lo_smem, 0);
    CUDA_CHECK(cudaDeviceSynchronize());
    CUDA_CHECK(cudaMemcpy(hf.data(), e->frames, sizeof(HzFrame) * hf.size(), cudaMemcpyDeviceToHost));
    cudaFree(d_stab);
    for (int k = 0; k < n; k++) {
        EncLane &l = e->lanes[(size_t) k];
        const HzFrame &f = hf[(size_t) k];
        /* as the engine: an overflowed packet is dirty up to its cap */
        l.pkt_dirty = f.overflow ? pics[k].cap - 64 : f.total_bytes;
        unsigned *info = info_out + 8 * k;
        info[0] = f.overflow;
        info[1] = f.total_bytes;
        for (int p = 0; p < 3; p++) {
            info[2 + p] = f.plane_bytes[p];
            info[5 + p] = (unsigned) sj[(size_t) 3 * k + p].dg.total;
        }
        CUDA_CHECK(cudaMemcpy(pkt_out + (e->pkt_bytes + DSVK_PKT_GUARD) * k, l.d_pkt, e->pkt_bytes + DSVK_PKT_GUARD, cudaMemcpyDeviceToHost));
        CUDA_CHECK(cudaMemcpy(coef_out + g.coef_total * k, l.coef, g.coef_total * sizeof(int32_t), cudaMemcpyDeviceToHost));
        for (int p = 0; p < 3; p++) {
            CUDA_CHECK(cudaMemcpy(dv_out + e->dv_pitch * (3 * k + p), l.dv[p], sbt_dv_elems(g.cw[p], g.ch[p]) * sizeof(int32_t),
                                  cudaMemcpyDeviceToHost));
        }
        CUDA_CHECK(cudaMemcpy(tflags_out + (size_t) g.total_tiles * k, l.tflags, (size_t) g.total_tiles, cudaMemcpyDeviceToHost));
        download_frame(l.recon[0], recon_out + g.frame_bytes * k);
    }
    return 0;
    DSV_API_END(-100)
}

/* the entropy-coding half of phase 3 on caller coefficients and caller tile flags: quantise + dequantise in place
 * (hzcc_quant_kernel, which the forward transform's epilogue does in the engine), then scan / prefix / pack with the
 * engine's list scratch and list modes.  Lets a caller place non-zeros at chosen scan positions and chunk edges. */
extern "C" int dsvk_hz_enc_batch(int w, int h, int subsamp, int blk_w, int blk_h, int n, const DSVK_PIC *pics, int32_t *coef_io,
                                 const uint8_t *tflags, uint8_t *pkt_out, unsigned *info_out, int32_t *dv_out)
{
    DSV_API_BEGIN
    if (w < 16 || h < 16 || (w & 1) || (h & 1) || n < 1) {
        return -1;
    }
    CodecGeom g;
    plan_geometry(&g, w, h, subsamp);
    plan_blocks(&g, blk_w, blk_h);
    const size_t pkt_bytes = enc_packet_cap(g), dv_pitch = sbt_dv_elems(g.cw[0], g.ch[0]);
    std::vector<SbtJob> sj((size_t) 3 * n);
    std::vector<HzJob> hj((size_t) 3 * n);
    std::vector<HzFrame> hf((size_t) n);
    std::vector<void *> bufs;
    auto keep = [&](void *p) { bufs.push_back(p); return p; };
    int n_p = 0;
    for (int k = 0; k < n; k++) {
        if (pics[k].cap > pkt_bytes || pics[k].start_byte + 64 > pics[k].cap) {
            for (void *b : bufs) {
                cudaFree(b);
            }
            return -1;
        }
        int32_t *coef = static_cast<int32_t *>(keep(dev_alloc<int32_t>(g.coef_total, false)));
        CUDA_CHECK(cudaMemcpy(coef, coef_io + g.coef_total * k, g.coef_total * sizeof(int32_t), cudaMemcpyHostToDevice));
        uint8_t *tf = nullptr;
        if (tflags) {
            tf = static_cast<uint8_t *>(keep(dev_alloc<uint8_t>((size_t) g.total_tiles)));
            CUDA_CHECK(cudaMemcpy(tf, tflags + (size_t) g.total_tiles * k, (size_t) g.total_tiles, cudaMemcpyHostToDevice));
        }
        uint8_t *dense = static_cast<uint8_t *>(keep(dev_alloc<uint8_t>((size_t) g.total_chunks * HZ_DENSE_BYTES, false)));
        uint8_t *stab = static_cast<uint8_t *>(keep(dev_alloc<uint8_t>((size_t) g.nblk, false)));
        CUDA_CHECK(cudaMemcpy(stab, pics[k].stable, (size_t) g.nblk, cudaMemcpyHostToDevice));
        uint8_t *pkt = static_cast<uint8_t *>(keep(dev_alloc<uint8_t>(pkt_bytes + DSVK_PKT_GUARD)));
        const int isP = pics[k].isP != 0;
        n_p += isP;
        for (int p = 0; p < 3; p++) {
            EncPlaneIO io;
            memset(&io, 0, sizeof(io));
            io.coef = coef + g.coef_off[p];
            io.dv = static_cast<int32_t *>(keep(dev_alloc<int32_t>(sbt_dv_elems(g.cw[p], g.ch[p]))));
            io.tflags = tf;
            io.hz_dense = dense;
            io.stable = stab;
            enc_fill_plane(&sj[(size_t) 3 * k + p], &hj[(size_t) 3 * k + p], g, p, k, isP, pics[k].quant, io);
        }
        enc_fill_frame(&hf[(size_t) k], pkt, pics[k].cap, pics[k].start_byte, k);
    }
    HzJob *d_hj = static_cast<HzJob *>(keep(dev_alloc<HzJob>(hj.size(), false)));
    HzFrame *d_hf = static_cast<HzFrame *>(keep(dev_alloc<HzFrame>(hf.size(), false)));
    HzChunk *d_ck = static_cast<HzChunk *>(keep(dev_alloc<HzChunk>((size_t) n * g.total_chunks, false)));
    CUDA_CHECK(cudaMemcpy(d_hj, hj.data(), sizeof(HzJob) * hj.size(), cudaMemcpyHostToDevice));
    CUDA_CHECK(cudaMemcpy(d_hf, hf.data(), sizeof(HzFrame) * hf.size(), cudaMemcpyHostToDevice));
    hzcc_quant_launch(d_hj, 3 * n, g.cw[0] * g.ch[0], 0);
    hzcc_enc_launch(d_hj, 3 * n, d_ck, n * g.total_chunks, d_hf, n, 0, g.total_chunks, g.chunks[0], g.chunks[1], n_p < n);
    CUDA_CHECK(cudaDeviceSynchronize());
    CUDA_CHECK(cudaMemcpy(hf.data(), d_hf, sizeof(HzFrame) * hf.size(), cudaMemcpyDeviceToHost));
    for (int k = 0; k < n; k++) {
        const HzFrame &f = hf[(size_t) k];
        unsigned *info = info_out + 8 * k;
        info[0] = f.overflow;
        info[1] = f.total_bytes;
        for (int p = 0; p < 3; p++) {
            const HzJob &hp = hj[(size_t) 3 * k + p];
            info[2 + p] = f.plane_bytes[p];
            info[5 + p] = (unsigned) hp.dg.total;
            CUDA_CHECK(cudaMemcpy(dv_out + dv_pitch * (3 * k + p), hp.dv, sbt_dv_elems(g.cw[p], g.ch[p]) * sizeof(int32_t),
                                  cudaMemcpyDeviceToHost));
        }
        CUDA_CHECK(cudaMemcpy(pkt_out + (pkt_bytes + DSVK_PKT_GUARD) * k, f.pkt, pkt_bytes + DSVK_PKT_GUARD, cudaMemcpyDeviceToHost));
        CUDA_CHECK(cudaMemcpy(coef_io + g.coef_total * k, hj[(size_t) 3 * k].coef, g.coef_total * sizeof(int32_t),
                              cudaMemcpyDeviceToHost));
    }
    for (void *b : bufs) {
        cudaFree(b);
    }
    return 0;
    DSV_API_END(-100)
}

/* the inverse transform of n pictures in one launch sequence, each picture with its own format */
extern "C" int dsvk_inv_batch(int n, const int *geo, const DSVK_PIC *pics, const int32_t *coef, const uint8_t *tflags,
                              const uint8_t *pred, uint8_t *out)
{
    DSV_API_BEGIN
    if (n < 1) {
        return -1;
    }
    std::vector<CodecGeom> g((size_t) n);
    std::vector<SbtJob> sj((size_t) 3 * n);
    std::vector<DevFrame> fo((size_t) n), fp((size_t) n);
    std::vector<void *> bufs;
    size_t lo_smem = 0;
    const int32_t *c_at = coef;
    const uint8_t *t_at = tflags, *p_at = pred;
    for (int k = 0; k < n; k++) {
        CodecGeom &gk = g[(size_t) k];
        if (geo[3 * k] < 16 || geo[3 * k + 1] < 16 || (geo[3 * k] & 1) || (geo[3 * k + 1] & 1)) {
            return -1;
        }
        plan_geometry(&gk, geo[3 * k], geo[3 * k + 1], geo[3 * k + 2]);
        plan_blocks(&gk, 16, 16);
        lo_smem = lo_smem > gk.lo_smem ? lo_smem : gk.lo_smem;
        devframe_alloc(&fo[(size_t) k], gk.w, gk.h, gk.subsamp);
        devframe_alloc(&fp[(size_t) k], gk.w, gk.h, gk.subsamp);
        if (pred) {
            upload_packed(fp[(size_t) k], p_at);
            p_at += gk.frame_bytes;
        }
        int32_t *dc = dev_alloc<int32_t>(gk.coef_total, false);
        CUDA_CHECK(cudaMemcpy(dc, c_at, gk.coef_total * sizeof(int32_t), cudaMemcpyHostToDevice));
        c_at += gk.coef_total;
        bufs.push_back(dc);
        uint8_t *dt = nullptr;
        if (tflags) {
            dt = dev_alloc<uint8_t>((size_t) gk.total_tiles);
            CUDA_CHECK(cudaMemcpy(dt, t_at, (size_t) gk.total_tiles, cudaMemcpyHostToDevice));
            t_at += gk.total_tiles;
            bufs.push_back(dt);
        }
        for (int p = 0; p < 3; p++) {
            int32_t *llx = dev_alloc<int32_t>(sbt_llx_elems(gk.cw[p], gk.ch[p]), false);
            bufs.push_back(llx);
            EncPlaneIO io;
            memset(&io, 0, sizeof(io));
            io.in = fo[(size_t) k].p[p];
            io.in_stride = fo[(size_t) k].stride[p];
            io.out = fo[(size_t) k].p[p];
            io.out_stride = fo[(size_t) k].stride[p];
            io.pred = pred ? fp[(size_t) k].p[p] : nullptr;
            io.pred_stride = fp[(size_t) k].stride[p];
            io.coef = dc + gk.coef_off[p];
            io.llx = llx;
            io.tflags = dt;
            HzJob unused;
            enc_fill_plane(&sj[(size_t) 3 * k + p], &unused, gk, p, k, pics[k].isP != 0, pics[k].quant, io);
        }
    }
    const SbtDims sdims = sbt_assign_tiles(sj.data(), 3 * n);
    SbtJob *d_sj = dev_alloc<SbtJob>(sj.size(), false);
    CUDA_CHECK(cudaMemcpy(d_sj, sj.data(), sizeof(SbtJob) * sj.size(), cudaMemcpyHostToDevice));
    sbt_inv_launch(d_sj, sdims, lo_smem, 0);
    CUDA_CHECK(cudaDeviceSynchronize());
    uint8_t *o_at = out;
    for (int k = 0; k < n; k++) {
        download_frame(fo[(size_t) k], o_at);
        o_at += g[(size_t) k].frame_bytes;
        devframe_free(&fo[(size_t) k]);
        devframe_free(&fp[(size_t) k]);
    }
    cudaFree(d_sj);
    for (void *b : bufs) {
        cudaFree(b);
    }
    return 0;
    DSV_API_END(-100)
}

/* dsvk_sse_batch / dsvk_ssim_batch: n picture pairs placed in bordered device frames, one launch of the kernel */
static int quality_batch(int n, const int *geo, const uint8_t *src, const uint8_t *rec, const uint8_t *border_fill, bool ssim, uint64_t *out)
{
    if (n < 1) {
        return -1;
    }
    std::vector<DevFrame> fs((size_t) n), fr((size_t) n);
    std::vector<SseJob> jobs((size_t) 3 * n);
    unsigned long long *d_out = dev_alloc<unsigned long long>((size_t) 3 * n);
    const uint8_t *s_at = src, *r_at = rec;
    int max_w = 0, max_h = 0;
    int rc = 0;
    for (int k = 0; k < n && rc == 0; k++) {
        if (geo[3 * k] < 16 || geo[3 * k + 1] < 16 || (geo[3 * k] & 1) || (geo[3 * k + 1] & 1)) {
            rc = -1;
            break;
        }
        CodecGeom g;
        plan_geometry(&g, geo[3 * k], geo[3 * k + 1], geo[3 * k + 2]);
        devframe_alloc(&fs[(size_t) k], g.w, g.h, g.subsamp);
        devframe_alloc(&fr[(size_t) k], g.w, g.h, g.subsamp);
        CUDA_CHECK(cudaMemset(fs[(size_t) k].alloc, border_fill[0], fs[(size_t) k].bytes));
        CUDA_CHECK(cudaMemset(fr[(size_t) k].alloc, border_fill[1], fr[(size_t) k].bytes));
        upload_packed(fs[(size_t) k], s_at);
        upload_packed(fr[(size_t) k], r_at);
        s_at += g.frame_bytes;
        r_at += g.frame_bytes;
        sse_fill_picture(&jobs[(size_t) 3 * k], g, fs[(size_t) k], fr[(size_t) k], d_out + 3 * k);
        max_w = max_w > g.w ? max_w : g.w;
        max_h = max_h > g.h ? max_h : g.h;
    }
    if (rc == 0) {
        SseJob *d_jobs = dev_alloc<SseJob>(jobs.size(), false);
        CUDA_CHECK(cudaMemcpy(d_jobs, jobs.data(), sizeof(SseJob) * jobs.size(), cudaMemcpyHostToDevice));
        if (ssim) {
            ssim_launch(d_jobs, 3 * n, max_w, max_h, 0);
        } else {
            sse_launch(d_jobs, 3 * n, max_h, 0);
        }
        CUDA_CHECK(cudaDeviceSynchronize());
        CUDA_CHECK(cudaMemcpy(out, d_out, sizeof(uint64_t) * 3 * n, cudaMemcpyDeviceToHost));
        cudaFree(d_jobs);
    }
    for (int k = 0; k < n; k++) {
        devframe_free(&fs[(size_t) k]);
        devframe_free(&fr[(size_t) k]);
    }
    cudaFree(d_out);
    return rc;
}

extern "C" int dsvk_sse_batch(int n, const int *geo, const uint8_t *src, const uint8_t *rec, const uint8_t *border_fill, uint64_t *sse_out)
{
    DSV_API_BEGIN
    return quality_batch(n, geo, src, rec, border_fill, false, sse_out);
    DSV_API_END(-100)
}

extern "C" int dsvk_ssim_batch(int n, const int *geo, const uint8_t *src, const uint8_t *rec, const uint8_t *border_fill,
                               int64_t *sum_out, int64_t *windows_out)
{
    DSV_API_BEGIN
    const int rc = quality_batch(n, geo, src, rec, border_fill, true, reinterpret_cast<uint64_t *>(sum_out));
    for (int k = 0; k < n && rc == 0; k++) {
        CodecGeom g;
        plan_geometry(&g, geo[3 * k], geo[3 * k + 1], geo[3 * k + 2]);
        for (int p = 0; p < 3; p++) {
            windows_out[3 * k + p] = ssim_windows(g.pw[p], g.ph[p]);
        }
    }
    return rc;
    DSV_API_END(-100)
}

/* one lane of DecEngine: coefficient planes and tile flags carry over from picture to picture */
struct DsvkDec {
    CodecGeom g;
    DecLane l;
};

extern "C" void *dsvk_dec_create(int w, int h, int subsamp, int blk_w, int blk_h)
{
    DSV_API_BEGIN
    if (w < 16 || h < 16 || (w & 1) || (h & 1)) {
        return nullptr;
    }
    DsvkDec *d = new DsvkDec;
    plan_geometry(&d->g, w, h, subsamp);
    plan_blocks(&d->g, blk_w, blk_h);
    dec_lane_alloc(d->l, d->g);
    return d;
    DSV_API_END(nullptr)
}

extern "C" void dsvk_dec_destroy(void *handle)
{
    DsvkDec *d = static_cast<DsvkDec *>(handle);
    if (!d) {
        return;
    }
    dec_lane_free(d->l);
    delete d;
}

/* the coefficient half of DecEngine::step on one picture: planes = the three plane records (32-bit plen, then the
 * plane's bytes) back to back, len bytes.  Returns the number of planes decoded. */
extern "C" int dsvk_dec_run(void *handle, const DSVK_PIC *pic, const uint8_t *planes, int len, int32_t *coef_out, uint8_t *tflags_out)
{
    DSV_API_BEGIN
    DsvkDec *d = static_cast<DsvkDec *>(handle);
    const CodecGeom &g = d->g;
    DecLane &l = d->l;
    if (len <= 0) {
        return -1;
    }
    uint8_t *d_pkt = dev_alloc<uint8_t>((size_t) len + 64);
    CUDA_CHECK(cudaMemcpy(d_pkt, planes, (size_t) len, cudaMemcpyHostToDevice));
    uint8_t *d_stab = dev_alloc<uint8_t>((size_t) g.nblk, false);
    CUDA_CHECK(cudaMemcpy(d_stab, pic->stable, (size_t) g.nblk, cudaMemcpyHostToDevice));
    HzPlaneData pd[3];
    const int nplanes = parse_plane_dir(planes, (unsigned) len, 0, g, d_pkt, pd);
    SbtJob sj[3];
    HzCleanItem clean[3];
    std::vector<uint8_t> hzj(hzdec_job_size() * 3);
    HzDecDims dims;
    for (int p = 0; p < 3; p++) {
        HzJob h;
        dec_fill_plane(&sj[p], &h, &clean[p], g, p, pic->isP != 0, pic->quant, l.out[l.cur], l.coef, l.llx[p], l.tflags, d_stab);
        if (p < nplanes) {
            hzdec_fill_job(hzj.data() + hzdec_job_size() * (size_t) dims.njobs, h, pd[p], l.hz[p], &dims);
        }
    }
    HzCleanItem *d_clean = dev_alloc<HzCleanItem>(3, false);
    void *d_hzj = dev_alloc<uint8_t>(hzj.size(), false);
    CUDA_CHECK(cudaMemcpy(d_clean, clean, sizeof(clean), cudaMemcpyHostToDevice));
    CUDA_CHECK(cudaMemcpy(d_hzj, hzj.data(), hzj.size(), cudaMemcpyHostToDevice));
    hzdec_clean_launch(d_clean, 3, g.tiles[0], 0);
    hzdec_launch_jobs(d_hzj, dims, 0);
    CUDA_CHECK(cudaDeviceSynchronize());
    CUDA_CHECK(cudaMemcpy(coef_out, l.coef, g.coef_total * sizeof(int32_t), cudaMemcpyDeviceToHost));
    CUDA_CHECK(cudaMemcpy(tflags_out, l.tflags, (size_t) g.total_tiles, cudaMemcpyDeviceToHost));
    cudaFree(d_pkt);
    cudaFree(d_stab);
    cudaFree(d_clean);
    cudaFree(d_hzj);
    return nplanes;
    DSV_API_END(-100)
}

/* ---- batch entry points: the motion kernels configured as the engines launch them --------------------------------- */

/* EncEngine's lanes for its phase 1: ingested frames and pyramids alternate with the picture parity (cur), so a lane's
 * search reference is its previous call's ingested frame */
struct DsvkMe {
    CodecGeom g;
    MotionGeom mg;
    int levels, max_pics;
    std::vector<EncLane> lanes;
    DevMV *d_mv0 = nullptr, *h_mv0 = nullptr; /* level-0 fields of all lanes, lane-major (EncEngine::d_mv0_ / h_mv0_) */
    uint8_t *d_stage = nullptr; /* staging of host pictures, one slot per lane (EncLane::d_in[0]) */
    LaneMisc *d_misc = nullptr;
    StepArena arena;
};

#define DSVK_STAGE_SLACK 256 /* bytes past a staged picture: host pictures may be staged at offsets 0..255 */

extern "C" void *dsvk_me_create(int w, int h, int subsamp, int blk_w, int blk_h, int levels, int max_pics)
{
    DSV_API_BEGIN
    if (w < 16 || h < 16 || (w & 1) || (h & 1) || levels < 1 || levels > DSV_MAX_PYRAMID_LEVELS || max_pics < 1 || blk_w < 1 || blk_h < 1) {
        return nullptr;
    }
    DsvkMe *m = new DsvkMe;
    plan_geometry(&m->g, w, h, subsamp);
    plan_blocks(&m->g, blk_w, blk_h);
    const CodecGeom &g = m->g;
    m->mg = motion_geom(g, levels);
    m->levels = levels;
    m->max_pics = max_pics;
    m->d_mv0 = dev_alloc<DevMV>((size_t) g.nblk * max_pics);
    CUDA_CHECK(cudaMallocHost(&m->h_mv0, sizeof(DevMV) * (size_t) g.nblk * max_pics));
    memset(m->h_mv0, 0, sizeof(DevMV) * (size_t) g.nblk * max_pics);
    m->d_misc = dev_alloc<LaneMisc>((size_t) max_pics);
    m->arena.create(((size_t) 3 * sizeof(IngestItem) + (size_t) levels * sizeof(Down2Item) + sizeof(SumItem) +
                     (size_t) (levels + 1) * sizeof(HmeArgs) + sizeof(BmcArgs) + 3 * sizeof(PlaneRef) + 256) * max_pics + 4096);
    /* slots start 256-byte aligned, as a buffer of their own would */
    const size_t stage_pitch = (g.frame_bytes + DSVK_STAGE_SLACK + 255) & ~(size_t) 255;
    CUDA_CHECK(cudaMalloc(&m->d_stage, stage_pitch * max_pics));
    m->lanes.resize((size_t) max_pics);
    for (int i = 0; i < max_pics; i++) {
        EncLane &l = m->lanes[(size_t) i];
        enc_lane_alloc(l, g, true, levels, enc_packet_cap(g));
        l.d_mvf[0] = m->d_mv0 + (size_t) i * g.nblk;
        l.d_in[0] = m->d_stage + stage_pitch * i;
    }
    return m;
    DSV_API_END(nullptr)
}

extern "C" void dsvk_me_destroy(void *handle)
{
    DsvkMe *m = static_cast<DsvkMe *>(handle);
    if (!m) {
        return;
    }
    for (auto &l : m->lanes) {
        enc_lane_free(l);
    }
    cudaFree(m->d_stage);
    cudaFree(m->d_mv0);
    cudaFreeHost(m->h_mv0);
    cudaFree(m->d_misc);
    m->arena.destroy();
    delete m;
}

extern "C" long dsvk_me_frame_bytes(void *handle, int level)
{
    const DsvkMe *m = static_cast<const DsvkMe *>(handle);
    if (level < 0 || level > m->levels) {
        return -1;
    }
    const EncLane &l = m->lanes[0];
    return (long) (level == 0 ? l.pad[0].bytes : l.pyr[0][level - 1].bytes);
}

/* phase 1 of EncEngine::step (encoder.cpp) and its motion compensation on pictures 0..n-1 in lanes 0..n-1 */
extern "C" int dsvk_me_run(void *handle, int n, const DSVK_ME_PIC *pics, const void *mvs, uint8_t *frames_out, int64_t *misc_out,
                           void *mv_out, uint8_t *pred_out, uint8_t *resid_out)
{
    DSV_API_BEGIN
    DsvkMe *m = static_cast<DsvkMe *>(handle);
    const CodecGeom &g = m->g;
    const MotionGeom &mg = m->mg;
    const int levels = m->levels;
    const bool code = mvs != nullptr;
    if (n < 1 || n > m->max_pics) {
        return -1;
    }
    int n_search = 0, n_sum = 0;
    for (int k = 0; k < n; k++) {
        if ((pics[k].has_ref && !m->lanes[(size_t) k].have_ref) || pics[k].stage_offset >= DSVK_STAGE_SLACK || !pics[k].src) {
            return -1;
        }
        n_search += pics[k].has_ref != 0;
        n_sum += pics[k].do_sum != 0;
    }
    StepArena &ar = m->arena;
    ar.reset();
    IngestItem *d_ing;
    IngestItem *ing = ar.push_n<IngestItem>((size_t) 3 * n, &d_ing);
    for (int k = 0; k < n; k++) {
        EncLane &l = m->lanes[(size_t) k];
        const uint8_t *base = pics[k].src;
        if (!pics[k].src_on_device) {
            uint8_t *stage = l.d_in[0] + pics[k].stage_offset;
            CUDA_CHECK(cudaMemcpy(stage, pics[k].src, g.frame_bytes, cudaMemcpyHostToDevice));
            base = stage;
        }
        const uint8_t *packed[3] = {base + g.plane_off[0], base + g.plane_off[1], base + g.plane_off[2]};
        ingest_fill_picture(&ing[3 * k], packed, l.pad[l.cur]);
    }
    Down2Item *d_dn[DSV_MAX_PYRAMID_LEVELS] = {};
    SumItem *d_sum = nullptr;
    HmeArgs *d_hme = nullptr;
    if (!code) {
        for (int lv = 0; lv < levels; lv++) {
            Down2Item *dn = ar.push_n<Down2Item>((size_t) n, &d_dn[lv]);
            for (int k = 0; k < n; k++) {
                EncLane &l = m->lanes[(size_t) k];
                down2_fill_level(&dn[k], l.pad[l.cur], l.pyr[l.cur], lv);
            }
        }
        if (n_sum) {
            SumItem *sm = ar.push_n<SumItem>((size_t) n_sum, &d_sum);
            for (int k = 0, q = 0; k < n; k++) {
                if (pics[k].do_sum) {
                    sum_fill_lane(&sm[q++], m->lanes[(size_t) k].pyr[m->lanes[(size_t) k].cur], levels, m->d_misc, k);
                }
            }
        }
        if (n_search) {
            HmeArgs *ha = ar.push_n<HmeArgs>((size_t) (levels + 1) * n_search, &d_hme);
            for (int k = 0, q = 0; k < n; k++) {
                EncLane &l = m->lanes[(size_t) k];
                if (pics[k].has_ref) {
                    hme_fill_lane(ha, n_search, q++, mg, l.pad[l.cur], l.pyr[l.cur], l.pad[l.cur ^ 1], l.pyr[l.cur ^ 1], l.d_mvf, l.d_aux,
                                  m->d_misc, k);
                }
            }
        }
    }
    BmcArgs *d_bmc = nullptr;
    if (n_search) {
        BmcArgs *ba = ar.push_n<BmcArgs>((size_t) n_search, &d_bmc);
        for (int k = 0, q = 0; k < n; k++) {
            EncLane &l = m->lanes[(size_t) k];
            if (pics[k].has_ref) {
                enc_bmc_fill(&ba[q++], mg, l.d_mvf[0], l.recon[l.cur ^ 1], l.pred, l.pad[l.cur], l.xf);
            }
        }
    }
    ZeroItem *d_zmisc;
    ZeroItem *zmisc = ar.push_n<ZeroItem>(1, &d_zmisc);
    zmisc->p = m->d_misc;
    zmisc->bytes = sizeof(LaneMisc) * (size_t) m->max_pics;
    PlaneRef *d_ext;
    PlaneRef *ext = ar.push_n<PlaneRef>((size_t) 3 * n, &d_ext);
    int n_ext = 0;
    for (int k = 0; k < n; k++) {
        if (pics[k].recon) {
            for (int p = 0; p < 3; p++) {
                ext[n_ext++] = plane_ref(m->lanes[(size_t) k].recon[m->lanes[(size_t) k].cur], p);
            }
        }
    }
    ar.upload(0);
    /* the launch sequence of EncEngine::step: search pass, or (code pass) the caller's vectors and the compensation */
    ingest_launch(d_ing, 3 * n, g.w, g.h, 0);
    if (code) {
        if (n_search) {
            for (int k = 0; k < n; k++) {
                if (pics[k].has_ref) {
                    memcpy(m->h_mv0 + (size_t) k * g.nblk, static_cast<const DevMV *>(mvs) + (size_t) k * g.nblk, sizeof(DevMV) * (size_t) g.nblk);
                }
            }
            copy1_launch(m->d_mv0, m->h_mv0, sizeof(DevMV) * (size_t) g.nblk * m->max_pics, 0);
            bmc_launch(d_bmc, n_search, mg, 0);
        }
    } else {
        for (int lv = 0; lv < levels; lv++) {
            down2_launch(d_dn[lv], n, ceil_shift(g.w, lv + 1), ceil_shift(g.h, lv + 1), 0);
        }
        if (n_sum || n_search) {
            zero_launch(d_zmisc, 1, zmisc->bytes, 0);
        }
        if (n_sum) {
            sum_launch(d_sum, n_sum, ceil_shift(g.h, levels), 0);
        }
        if (n_search) {
            hme_launch(d_hme, n_search, mg, 0);
            bmc_launch(d_bmc, n_search, mg, 0);
        }
    }
    CUDA_CHECK(cudaDeviceSynchronize());
    /* phase 3's new reference: the caller's reconstruction, bordered */
    for (int k = 0; k < n; k++) {
        if (pics[k].recon) {
            upload_packed(m->lanes[(size_t) k].recon[m->lanes[(size_t) k].cur], pics[k].recon);
        }
    }
    if (n_ext) {
        extend_launch(d_ext, n_ext, g.w, g.h, 0);
    }
    CUDA_CHECK(cudaDeviceSynchronize());
    std::vector<LaneMisc> misc((size_t) n);
    CUDA_CHECK(cudaMemcpy(misc.data(), m->d_misc, sizeof(LaneMisc) * (size_t) n, cudaMemcpyDeviceToHost));
    CUDA_CHECK(cudaMemcpy(mv_out, m->d_mv0, sizeof(DevMV) * (size_t) g.nblk * n, cudaMemcpyDeviceToHost));
    uint8_t *f_at = frames_out;
    for (int k = 0; k < n; k++) {
        EncLane &l = m->lanes[(size_t) k];
        misc_out[2 * k] = (int64_t) misc[(size_t) k].luma_sum;
        misc_out[2 * k + 1] = misc[(size_t) k].nintra;
        CUDA_CHECK(cudaMemcpy(f_at, l.pad[l.cur].alloc, l.pad[l.cur].bytes, cudaMemcpyDeviceToHost));
        f_at += l.pad[l.cur].bytes;
        for (int lv = 0; lv < levels; lv++) {
            CUDA_CHECK(cudaMemcpy(f_at, l.pyr[l.cur][lv].alloc, l.pyr[l.cur][lv].bytes, cudaMemcpyDeviceToHost));
            f_at += l.pyr[l.cur][lv].bytes;
        }
        download_frame(l.pred, pred_out + g.frame_bytes * k);
        download_frame(l.xf, resid_out + g.frame_bytes * k);
        l.have_ref = 1;
        l.cur ^= 1;
    }
    return 0;
    DSV_API_END(-100)
}

/* the compensation of DecEngine::step (decoder.cpp) on n lanes: resid[k] is lane k's inverse-transform output, ref[k] its
 * previous picture (bordered as the decoder's step leaves it); only the P lanes are in the launch's list */
extern "C" int dsvk_add_pred_batch(int w, int h, int subsamp, int blk_w, int blk_h, int n, const int *isP, const void *mvs,
                                   const uint8_t *resid, const uint8_t *ref, uint8_t *out)
{
    DSV_API_BEGIN
    if (w < 16 || h < 16 || (w & 1) || (h & 1) || n < 1 || blk_w < 1 || blk_h < 1) {
        return -1;
    }
    CodecGeom g;
    plan_geometry(&g, w, h, subsamp);
    plan_blocks(&g, blk_w, blk_h);
    const MotionGeom mg = motion_geom(g, 0);
    std::vector<DevFrame> cur((size_t) n), prev((size_t) n);
    DevMV *d_mv = dev_alloc<DevMV>((size_t) g.nblk * n, false);
    CUDA_CHECK(cudaMemcpy(d_mv, mvs, sizeof(DevMV) * (size_t) g.nblk * n, cudaMemcpyHostToDevice));
    std::vector<BmcArgs> ba((size_t) n);
    int n_p = 0;
    for (int k = 0; k < n; k++) {
        devframe_alloc(&cur[(size_t) k], w, h, subsamp);
        devframe_alloc(&prev[(size_t) k], w, h, subsamp);
        upload_packed(cur[(size_t) k], resid + g.frame_bytes * k);
        upload_packed(prev[(size_t) k], ref + g.frame_bytes * k);
        frame_extend_launch(prev[(size_t) k], 3, 0);
        dec_bmc_fill(ba.data(), &n_p, isP[k] != 0, mg, d_mv, k, g.nblk, prev[(size_t) k], cur[(size_t) k]);
    }
    BmcArgs *d_ba = dev_alloc<BmcArgs>((size_t) n, false);
    CUDA_CHECK(cudaMemcpy(d_ba, ba.data(), sizeof(BmcArgs) * (size_t) n_p, cudaMemcpyHostToDevice));
    bmc_launch(d_ba, n_p, mg, 0);
    CUDA_CHECK(cudaDeviceSynchronize());
    for (int k = 0; k < n; k++) {
        download_frame(cur[(size_t) k], out + g.frame_bytes * k);
        devframe_free(&cur[(size_t) k]);
        devframe_free(&prev[(size_t) k]);
    }
    cudaFree(d_ba);
    cudaFree(d_mv);
    return 0;
    DSV_API_END(-100)
}
