/*
 * quality.cu -- per-plane squared error and SSIM between a source and its reconstruction (no reference counterpart:
 * the reference encoder measures no distortion).  The batch encoders' per-picture reports (dsvb_enc_picture_info,
 * dsvb_enc_picture_ssim) and the kernel-level dsvk_sse_batch / dsvk_ssim_batch launch them over every plane of every
 * picture of a step at once.
 *
 * Both operands are bordered DevFrame planes: rows start 16-byte aligned and strides are multiples of 16
 * (frame.cuh), so a thread reads 16 samples of each with one load.  The bytes of the last chunk of a row past pw
 * are border or padding, which differ between the two frames; they are masked out.
 */
#include <cmath>

#include "frame.cuh"

namespace dsv {

#define SSE_WARPS 8
#define SSE_ROWS_PER_WARP 4 /* rows of one warp per block: fewer 64-bit atomics per plane */

DSV_D unsigned keep_low_bytes(int n) /* mask of the n (clamped to 0..4) low bytes of a word */
{
    return n >= 4 ? 0xffffffffu : n <= 0 ? 0u : (1u << (8 * n)) - 1u;
}

/* grid: x = bands of SSE_WARPS * SSE_ROWS_PER_WARP rows, y = job */
__global__ void __launch_bounds__(SSE_WARPS * 32) sse_kernel(const SseJob *jobs)
{
    const SseJob j = jobs[blockIdx.y];
    const int lane = (int) threadIdx.x & 31, warp = (int) threadIdx.x >> 5;
    const int nck = (j.pw + 15) >> 4;
    const int y0 = (int) blockIdx.x * SSE_WARPS * SSE_ROWS_PER_WARP + warp;
    unsigned long long acc = 0;
    for (int r = 0; r < SSE_ROWS_PER_WARP; r++) {
        const int y = y0 + r * SSE_WARPS;
        if (y >= j.ph) {
            break; /* uniform across the warp */
        }
        const uint4 *s = reinterpret_cast<const uint4 *>(j.src + (size_t) y * j.src_stride);
        const uint4 *q = reinterpret_cast<const uint4 *>(j.rec + (size_t) y * j.rec_stride);
        /* 32-bit partial sum over one row: a lane loads at most ceil(16384 / 16 / 32) = 32 chunks of 16 samples,
         * 32 * 16 * 255^2 < 2^26 */
        unsigned row = 0;
        for (int c = lane; c < nck; c += 32) {
            const uint4 a = s[c], b = q[c];
            unsigned d0 = __vabsdiffu4(a.x, b.x), d1 = __vabsdiffu4(a.y, b.y), d2 = __vabsdiffu4(a.z, b.z), d3 = __vabsdiffu4(a.w, b.w);
            const int left = j.pw - 16 * c; /* samples of this chunk inside the plane */
            if (left < 16) {
                d0 &= keep_low_bytes(left);
                d1 &= keep_low_bytes(left - 4);
                d2 &= keep_low_bytes(left - 8);
                d3 &= keep_low_bytes(left - 12);
            }
            row = __dp4a(d0, d0, row);
            row = __dp4a(d1, d1, row);
            row = __dp4a(d2, d2, row);
            row = __dp4a(d3, d3, row);
        }
        acc += row;
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        acc += __shfl_xor_sync(0xffffffffu, acc, o);
    }
    if (lane == 0 && acc) {
        atomicAdd(j.out, acc); /* integer sums: exact and independent of the order */
    }
}

void sse_launch(const SseJob *d_jobs, int n, int max_h, cudaStream_t st)
{
    if (n > 0 && max_h > 0) {
        DSV_LAUNCH(sse_kernel, dim3((unsigned) ceil_div(max_h, SSE_WARPS * SSE_ROWS_PER_WARP), (unsigned) n), dim3(SSE_WARPS * 32), 0, st,
                   d_jobs);
        KERNEL_CHECK();
    }
}

/*
 * SSIM as x264 / ffmpeg define it for 8-bit samples (include/dsv1_b200_batch.h, DSVB_PICSSIM): sums over 4x4 blocks,
 * 8x8 windows made of 2x2 blocks at a stride of 4 samples, integer constants.  Each window's value is rounded to a
 * multiple of 2^-32 and the plane sums those integers, so the result does not depend on the order of the sums.
 *
 * A CTA owns a tile of SSIM_TW x SSIM_TH windows and keeps the sums of the (SSIM_TW + 1) x (SSIM_TH + 1) blocks
 * they cover in shared memory: the blocks of the next tile's first column and row are read twice.  Shared memory
 * does not depend on the plane's width.
 *   phase 1: a thread reads 4 rows of a 16-sample chunk of both planes (16-byte loads) and forms the sums of its 4
 *            blocks with __dp4a; the tile's rows are 32 chunks wide plus one chunk for the halo column (of which one
 *            block is used).  Blocks past bw read border or padding bytes, which differ between the frames; no window
 *            uses them.
 *   phase 2: two threads per window column walk down SSIM_TH / 2 windows each, adding the horizontal pair sums of two
 *            block rows; the windows' integer values are summed per warp and added with one 64-bit atomic.
 */
#define SSIM_THREADS 256
#define SSIM_TW 128 /* window columns of a tile: 32 chunks of 4 blocks */
#define SSIM_TH 14  /* window rows of a tile: 33 chunks x 15 block rows = 495 chunk loads, two rounds of 256 threads */
#define SSIM_BW (SSIM_TW + 4)
#define SSIM_BH (SSIM_TH + 1)

/* rint(ssim * 2^32) of one window from its sums: s1 = sum a, s2 = sum b, ss = sum (a^2 + b^2), s12 = sum ab over 64
 * samples.  Every factor fits 32 bits (s1, s2 <= 16320, 64 * ss <= 532684800, |covar| <= 266342400); the two
 * products are formed in 64 bits, exactly as the definition's int64 arithmetic. */
DSV_D long long ssim_window_q32(int s1, int s2, int ss, int s12)
{
    const int vars = 64 * ss - s1 * s1 - s2 * s2;
    const int covar = 64 * s12 - s1 * s2;
    const long long num = (long long) (2 * s1 * s2 + 416) * (long long) (2 * covar + 235963);
    const long long den = (long long) (s1 * s1 + s2 * s2 + 416) * (long long) (vars + 235963);
    /* IEEE division; llrint rounds half to even (the device's default rounding mode; cvt.rni.s64.f64) */
    return llrint((double) num / (double) den * 4294967296.0);
}

/* grid: x = tiles across, y = tiles down (both sized for the widest / tallest plane), z = job */
__global__ void __launch_bounds__(SSIM_THREADS) ssim_kernel(const SseJob *jobs)
{
    const SseJob j = jobs[blockIdx.z];
    const int bw = j.pw >> 2, bh = j.ph >> 2;
    const int i0 = (int) blockIdx.x * SSIM_TW, j0 = (int) blockIdx.y * SSIM_TH; /* first block (= window) of the tile */
    if (i0 >= bw - 1 || j0 >= bh - 1) {
        return; /* no window of this plane in the tile: the whole CTA leaves */
    }
    /* block sums: [0] sum a, [1] sum b, [2] sum a^2 + b^2, [3] sum ab; at most 16 * 2 * 255^2 */
    __shared__ __align__(16) unsigned s_blk[4][SSIM_BH][SSIM_BW];
    const int nbx = min(SSIM_TW + 1, bw - i0), nby = min(SSIM_TH + 1, bh - j0); /* blocks the tile's windows cover */
    const int nck = (nbx + 3) >> 2;
    const size_t x0 = (size_t) 4 * i0;
    for (int t = (int) threadIdx.x; t < nck * nby; t += SSIM_THREADS) {
        const int r = t / nck, c = t - r * nck;
        const size_t y = (size_t) 4 * (j0 + r);
        unsigned sa[4] = {0, 0, 0, 0}, sb[4] = {0, 0, 0, 0}, ss[4] = {0, 0, 0, 0}, sab[4] = {0, 0, 0, 0};
#pragma unroll
        for (int dy = 0; dy < 4; dy++) {
            const uint4 a = *reinterpret_cast<const uint4 *>(j.src + (y + dy) * j.src_stride + x0 + 16 * c);
            const uint4 b = *reinterpret_cast<const uint4 *>(j.rec + (y + dy) * j.rec_stride + x0 + 16 * c);
            const unsigned wa[4] = {a.x, a.y, a.z, a.w}, wb[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int q = 0; q < 4; q++) {
                sa[q] = __dp4a(wa[q], 0x01010101u, sa[q]);
                sb[q] = __dp4a(wb[q], 0x01010101u, sb[q]);
                ss[q] = __dp4a(wa[q], wa[q], __dp4a(wb[q], wb[q], ss[q]));
                sab[q] = __dp4a(wa[q], wb[q], sab[q]);
            }
        }
        *reinterpret_cast<uint4 *>(&s_blk[0][r][4 * c]) = make_uint4(sa[0], sa[1], sa[2], sa[3]);
        *reinterpret_cast<uint4 *>(&s_blk[1][r][4 * c]) = make_uint4(sb[0], sb[1], sb[2], sb[3]);
        *reinterpret_cast<uint4 *>(&s_blk[2][r][4 * c]) = make_uint4(ss[0], ss[1], ss[2], ss[3]);
        *reinterpret_cast<uint4 *>(&s_blk[3][r][4 * c]) = make_uint4(sab[0], sab[1], sab[2], sab[3]);
    }
    __syncthreads();
    const int i = (int) threadIdx.x % SSIM_TW;
    const int r0 = (int) threadIdx.x / SSIM_TW * (SSIM_TH / 2), r1 = min(r0 + SSIM_TH / 2, nby - 1);
    long long acc = 0;
    if (i < nbx - 1 && r0 < r1) {
        unsigned up[4];
#pragma unroll
        for (int v = 0; v < 4; v++) {
            up[v] = s_blk[v][r0][i] + s_blk[v][r0][i + 1];
        }
        for (int r = r0; r < r1; r++) {
            unsigned dn[4];
#pragma unroll
            for (int v = 0; v < 4; v++) {
                dn[v] = s_blk[v][r + 1][i] + s_blk[v][r + 1][i + 1];
            }
            acc += ssim_window_q32((int) (up[0] + dn[0]), (int) (up[1] + dn[1]), (int) (up[2] + dn[2]), (int) (up[3] + dn[3]));
#pragma unroll
            for (int v = 0; v < 4; v++) {
                up[v] = dn[v];
            }
        }
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        acc += __shfl_xor_sync(0xffffffffu, acc, o);
    }
    if ((threadIdx.x & 31) == 0 && acc) {
        atomicAdd(j.out, (unsigned long long) acc); /* two's complement: negative sums wrap correctly */
    }
}

void ssim_launch(const SseJob *d_jobs, int n, int max_pw, int max_ph, cudaStream_t st)
{
    if (n > 0) {
        const int tx = ceil_div(imax(max_pw / 4 - 1, 1), SSIM_TW), ty = ceil_div(imax(max_ph / 4 - 1, 1), SSIM_TH);
        DSV_LAUNCH(ssim_kernel, dim3((unsigned) tx, (unsigned) ty, (unsigned) n), dim3(SSIM_THREADS), 0, st, d_jobs);
        KERNEL_CHECK();
    }
}

} // namespace dsv
