/*
 * frame.cuh -- device frames in the reference's bordered layout (frame.c:63-120): three u8 planes in one
 * allocation, 64-sample replicated border on every side, stride = roundup16(w + 128), planes back to
 * back.  Keeping the exact layout means in-bounds-but-past-border reads of the motion search / half-pel
 * filters (SURVEY.md Appendix B-9) see the same bytes as the reference; a zeroed guard band in front of
 * and behind the allocation makes the few reads that leave the reference's allocation well defined.
 *
 * All frame-level kernels are BATCHED: a launch takes a device array of small descriptors ("lists"), one
 * entry per plane (or plane pair) of every frame in flight, so that the lanes of a lock-step batch
 * (sequences x planes) share one grid.  Lists are assembled by the host in a StepArena and uploaded with a
 * single copy per pipeline phase.
 */
#pragma once
#include "common.cuh"

namespace dsv {

struct DevFrame {
    uint8_t *alloc = nullptr; /* cudaMalloc'd block incl. guards */
    uint8_t *p[3] = {nullptr, nullptr, nullptr}; /* sample (0,0) of each plane */
    int stride[3] = {0, 0, 0};
    int w[3] = {0, 0, 0}, h[3] = {0, 0, 0};
    size_t bytes = 0;
};

#define DSV_GUARD_BYTES (4 * 4096)

void devframe_alloc(DevFrame *f, int width, int height, int subsamp);
void devframe_free(DevFrame *f);

/* one bordered plane */
struct PlaneRef {
    uint8_t *p;
    int stride, w, h;
};
static inline PlaneRef plane_ref(const DevFrame &f, int c)
{
    PlaneRef r;
    r.p = f.p[c];
    r.stride = f.stride[c];
    r.w = f.w[c];
    r.h = f.h[c];
    return r;
}

/* list entries */
struct IngestItem { /* packed (dense, stride == w) plane -> bordered plane, border replicated */
    const uint8_t *src;
    PlaneRef dst;
};
struct PackItem { /* bordered plane -> packed plane */
    PlaneRef src;
    uint8_t *dst;
};
struct Down2Item { /* 2x2 rounded box filter of src -> dst, border replicated */
    PlaneRef src, dst;
};
struct SumItem { /* sum of all samples -> *out (zeroed by the host side of the launch) */
    PlaneRef src;
    unsigned long long *out;
};
struct ZeroItem { /* clear `bytes` bytes at p (16-byte aligned): done by a kernel, NOT cudaMemsetAsync, because memsets
                    run on a copy engine and would queue behind the large PCIe transfers of the copy stream */
    void *p;
    size_t bytes;
};
struct CopyItem { /* control-plane data moved by SMs through mapped pinned host memory (zero copy): the DMA engines stay
                    free for the bulk picture traffic of the copy stream, behind which engine copies would queue */
    void *dst;
    const void *src;
    size_t bytes;
};
struct SseJob { /* *out += sum over the pw x ph samples of (src - rec)^2 (quality.cu); both planes bordered DevFrame planes.
                  ssim_kernel takes the same jobs and adds the plane's sum of rint(ssim_w * 2^32) to *out (two's complement) */
    const uint8_t *src;
    const uint8_t *rec;
    int src_stride, rec_stride;
    int pw, ph;
    unsigned long long *out;
};
struct DevMV;
struct DrawItem { /* debug overlay (overlay.cu) painted in place on a picture whose three planes are dense */
    uint8_t *dst[3];
    int stride[3], w[3], h[3];
    const DevMV *mvs;
    const uint8_t *stab;
    int blk_w, blk_h, nbh, nbv;
    int mode; /* DSV_DRAW_* bits (dsv_decoder.h:38-40) */
};
struct To420Item { /* chroma plane -> dense 4:2:0 chroma plane of dw x dh samples (out420.cu) */
    PlaneRef src;
    uint8_t *dst;
    int dw, dh;
    int hpass; /* 1: 4:4:4 source (horizontal then vertical pass), 0: vertical pass only */
};

/*
 * Host-assembled, device-mirrored scratch for one pipeline phase: the host appends descriptor arrays into
 * pinned memory, gets back the address the same bytes will have on the device, and uploads everything
 * with one cudaMemcpyAsync before the launches that read it.
 */
struct StepArena {
    uint8_t *h = nullptr, *d = nullptr;
    size_t cap = 0, used = 0, uploaded = 0;
    void create(size_t bytes);
    void destroy();
    void reset() { used = uploaded = 0; }
    /* returns host pointer; *dev receives the device twin */
    void *push(size_t bytes, void **dev);
    template <typename T> T *push_n(size_t n, T **dev)
    {
        void *dv;
        T *hp = reinterpret_cast<T *>(push(n * sizeof(T), &dv));
        *dev = reinterpret_cast<T *>(dv);
        return hp;
    }
    void upload(cudaStream_t st); /* everything appended since the last upload */
    /* the same upload as a copy item for copyn_launch (marks it done); false: nothing is pending */
    bool take_upload(struct CopyItem *it);
};

/* launches; every list pointer is a DEVICE pointer, max_* bound the grid */
void ingest_launch(const IngestItem *d_items, int n, int max_w, int max_h, cudaStream_t st);
void pack_launch(const PackItem *d_items, int n, int max_w, int max_h, cudaStream_t st);
void extend_launch(const PlaneRef *d_items, int n, int max_w, int max_h, cudaStream_t st);
void down2_launch(const Down2Item *d_items, int n, int max_w, int max_h, cudaStream_t st);
void sum_launch(const SumItem *d_items, int n, int max_h, cudaStream_t st);
void zero_launch(const ZeroItem *d_items, int n, size_t max_bytes, cudaStream_t st);
/* items may live in mapped pinned host memory; one of dst/src of every item is device memory, the other may be
 * mapped pinned host memory */
void copy_launch(const CopyItem *items, int n, size_t max_bytes, cudaStream_t st);
void copy1_launch(void *dst, const void *src, size_t bytes, cudaStream_t st);
/* up to COPYN_MAX independent control-plane copies in ONE launch (each launch that reads mapped host memory costs a PCIe
 * round trip of ~14 us on the stream); items (host array) with bytes == 0 are skipped */
#define COPYN_MAX 4
void copyn_launch(const CopyItem *items, int n, cudaStream_t st);
void overlay_launch(const DrawItem *d_items, int n, cudaStream_t st);
void to420_launch(const To420Item *d_items, int n, int max_dw, int max_dh, cudaStream_t st);
/* squared error of every job's plane in ONE launch; the outputs must be zeroed before (quality.cu) */
void sse_launch(const SseJob *d_jobs, int n, int max_h, cudaStream_t st);
/* SSIM window sums of every job's plane in ONE launch (one launch even when no plane has a window); the outputs must be
 * zeroed before (quality.cu) */
void ssim_launch(const SseJob *d_jobs, int n, int max_pw, int max_ph, cudaStream_t st);

/* single-frame conveniences used by the kernel-level API (kernel_api.cu) */
void frame_extend_launch(const DevFrame &f, int nplanes, cudaStream_t st);
void frame_down2_luma_launch(const DevFrame &src, const DevFrame &dst, cudaStream_t st);

} // namespace dsv
