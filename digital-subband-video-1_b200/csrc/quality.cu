/*
 * quality.cu -- per-plane squared error between a source and its reconstruction (no reference counterpart: the
 * reference encoder measures no distortion).  The batch encoder's per-picture report (dsvb_enc_picture_info) and the
 * kernel-level dsvk_sse_batch launch it over every plane of every picture of a step at once.
 *
 * Both operands are bordered DevFrame planes: rows start 16-byte aligned and strides are multiples of 16
 * (frame.cuh), so a thread reads 16 samples of each with one load.  The bytes of the last chunk of a row past pw
 * are border or padding, which differ between the two frames; they are masked out.
 */
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

} // namespace dsv
