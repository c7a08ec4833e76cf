/*
 * engine.h -- lock-step batch engines behind both public APIs.
 *
 * An engine owns L "lanes" (independent sequences, each with its own reference frames, coefficient planes,
 * packet buffer and rate/stability state) and advances all active lanes by one picture per step(): every
 * pipeline stage is ONE kernel launch over the planes / blocks / chunks of all lanes, host<->device
 * synchronisation happens a fixed number of times per step regardless of L.
 *   dsv_enc / dsv_dec (dsv1_b200.h)          = an engine with one lane, one step per call
 *   dsvb_encode / dsvb_decode (dsv1_b200_batch.h) = L lanes, closed-GOP / whole-sequence sharding
 */
#pragma once
#include <time.h>

#include <atomic>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <thread>
#include <vector>

#include "dsv1_b200.h"
#include "dsv1_b200_batch.h"

#include "../frame.cuh"
#include "../hzcc.cuh"
#include "../hzcc_dec.cuh"
#include "../motion.cuh"
#include "../sbt.cuh"

namespace dsv {

struct CodecGeom {
    int w, h, subsamp, hs, vs;
    int pw[3], ph[3]; /* plane sizes */
    int cw[3], ch[3]; /* coefficient plane sizes (frame.c:29-61) */
    size_t coef_off[3], coef_total;
    size_t frame_bytes; /* packed planar frame */
    size_t plane_off[3];
    int blk_w, blk_h, nbh, nbv, nblk;
    int tiles[3], total_tiles;   /* SBT tiles per plane / picture */
    int chunks[3], total_chunks; /* HZCC encoder chunks per plane / picture */
    size_t lo_smem;
};

void plan_geometry(CodecGeom *g, int w, int h, int subsamp);
void plan_blocks(CodecGeom *g, int blk_w, int blk_h);
/* the motion kernels' view of a planned block grid, with `levels` pyramid levels */
MotionGeom motion_geom(const CodecGeom &g, int levels);
int size4dim(int dim);
void predict_mv(const DevMV *mvs, int nbh, int x, int y, int *px, int *py);

/* per-plane job descriptors of picture k of a step (plane_jobs.cpp): the engines and the kernel-level batch entry
 * points (kernel_api.cu) fill them with the same code */
struct EncPlaneIO {
    const uint8_t *in; /* forward input: the picture (I) or its residual (P) */
    int in_stride;
    uint8_t *out; /* the inverse's reconstruction */
    int out_stride;
    const uint8_t *pred; /* P pictures: prediction the inverse adds on its way out */
    int pred_stride;
    int32_t *coef, *llx, *dv; /* this plane's */
    uint8_t *tflags, *hz_dense; /* the picture's, all three planes */
    const uint8_t *stable;
};
void enc_fill_plane(SbtJob *s, HzJob *h, const CodecGeom &g, int p, int k, int isP, int quant, const EncPlaneIO &io);
/* bytes of a lane's packet buffer: the largest coded picture of the format plus its head */
size_t enc_packet_cap(const CodecGeom &g);
void enc_fill_frame(HzFrame *f, uint8_t *pkt, unsigned cap, unsigned start_byte, int k);
/* squared-error jobs of the three planes of a picture: out[p] receives plane p's sum */
void sse_fill_picture(SseJob *j, const CodecGeom &g, const DevFrame &src, const DevFrame &rec, unsigned long long *out);
/* SSIM windows of a pw x ph plane: (pw/4 - 1) * (ph/4 - 1), 0 when either factor is below 1 */
int64_t ssim_windows(int pw, int ph);
void dec_fill_plane(SbtJob *s, HzJob *h, HzCleanItem *c, const CodecGeom &g, int p, int isP, int quant, const DevFrame &cur,
                    int32_t *coef, int32_t *llx, uint8_t *tflags, const uint8_t *stable);
/* a lane's decoder tile flags before its first picture: every tile at the plane's base value (hz_flag_base) */
void dec_init_flags(uint8_t *d_tflags, const CodecGeom &g);

/* per-lane scalars of the encoder's phase 1, one record per lane in a lane-major device array */
struct LaneMisc {
    unsigned long long luma_sum;
    int nintra;
    int pad;
};
/* motion descriptors of one picture of a step (plane_jobs.cpp), filled the same way by the encode / decode engines and
 * by the kernel-level motion entry points (kernel_api.cu).  `pyr` is a lane's pyramid, levels 1.. of `top`. */
/* ingest of the three packed planes src[p] into the bordered frame dst */
void ingest_fill_picture(IngestItem *it, const uint8_t *const src[3], const DevFrame &dst);
/* pyramid level lv + 1 from level lv (lv = 0: the ingested frame) */
void down2_fill_level(Down2Item *it, const DevFrame &top, const DevFrame *pyr, int lv);
/* luma sum of the smallest level into misc[lane] */
void sum_fill_lane(SumItem *it, const DevFrame *pyr, int levels, LaneMisc *d_misc, int lane);
/* the levels + 1 search rows of lane slot q: rows[level * n_search + q]; the intra count goes to misc[lane] */
void hme_fill_lane(HmeArgs *rows, int n_search, int q, const MotionGeom &mg, const DevFrame &src, const DevFrame *src_pyr,
                   const DevFrame &ref, const DevFrame *ref_pyr, DevMV *const *mvf, int2 *aux, LaneMisc *d_misc, int lane);
/* encoder: prediction from the previous reconstruction into pred, residual of the ingested source into resid */
void enc_bmc_fill(BmcArgs *a, const MotionGeom &mg, const DevMV *mv, const DevFrame &recon_ref, const DevFrame &pred,
                  const DevFrame &src, const DevFrame &resid);
/* decoder: lane li's compensation, appended to list[*n_p] when the picture is P: in place on cur, no prediction kept;
 * the lane's vectors are at d_mv + li * nblk */
void dec_bmc_fill(BmcArgs *list, int *n_p, int isP, const MotionGeom &mg, const DevMV *d_mv, int li, int nblk, const DevFrame &ref,
                  const DevFrame &cur);

/* where one input / output picture lives */
struct PicRef {
    const uint8_t *plane[3];
    int stride[3];
    int on_device;
};

/* live timing of the dominant kernels (CUDA events on the engine's stream) + work counters */
struct EngineStats {
    double sbt_fwd_ms = 0, sbt_inv_ms = 0;
    unsigned long long sbt_fwd_launches = 0, sbt_inv_launches = 0;
    unsigned long long sbt_fwd_bytes = 0, sbt_inv_bytes = 0; /* algorithmic: w*h + 4*cw*ch per plane */
    double bmc_ms = 0;
    unsigned long long bmc_launches = 0, bmc_bytes = 0; /* algorithmic: 4 B per sample (encoder), 3 (decoder) */
    unsigned long long kernel_launches = 0;
    unsigned long long h2d_bytes = 0, d2h_bytes = 0;
    unsigned long long pictures = 0;
    double host_ms = 0; /* serial host work inside the steps (side info, packet heads, parsing) */
};

/* persistent worker threads for the per-lane serial host work of a step (side info, packet heads): lanes are
 * independent, so phase 2 of a 32-lane step need not be 32x the single-lane time while the GPU waits */
class HostPool {
public:
    explicit HostPool(int nthreads)
    {
        for (int i = 0; i < nthreads; i++) {
            th_.emplace_back([this] { worker(); });
        }
    }
    ~HostPool()
    {
        {
            std::lock_guard<std::mutex> lk(m_);
            quit_ = true;
        }
        cv_.notify_all();
        for (auto &t : th_) {
            t.join();
        }
    }
    void run(int n, const std::function<void(int)> &f)
    {
        if (th_.empty() || n <= 1) {
            for (int i = 0; i < n; i++) {
                f(i);
            }
            return;
        }
        unsigned long long ep;
        {
            std::lock_guard<std::mutex> lk(m_);
            fn_ = &f;
            n_ = n;
            ep = ++epoch_;
            pending_.store(n);
            next_.store(ep << 32); /* published last: index 0 of this epoch */
        }
        cv_.notify_all();
        drain(ep, n, &f);
        std::unique_lock<std::mutex> lk(m_);
        cv_done_.wait(lk, [this] { return pending_.load() == 0; });
        fn_ = nullptr;
    }

private:
    /* Items are claimed by compare-and-swap on (epoch << 32 | next index): a worker that is still leaving the
     * previous job when the next one is published cannot claim anything with its stale epoch, job size or function
     * (it took all three together under the mutex), so no index runs twice and none is lost. */
    void drain(unsigned long long ep, int n, const std::function<void(int)> *fn)
    {
        for (;;) {
            unsigned long long cur = next_.load();
            for (;;) {
                if ((cur >> 32) != ep || (int) (cur & 0xffffffffull) >= n) {
                    return;
                }
                if (next_.compare_exchange_weak(cur, cur + 1)) {
                    break;
                }
            }
            (*fn)((int) (cur & 0xffffffffull));
            if (pending_.fetch_sub(1) == 1) {
                std::lock_guard<std::mutex> lk(m_);
                cv_done_.notify_all();
            }
        }
    }
    void worker()
    {
        unsigned long long seen = 0;
        for (;;) {
            int n;
            const std::function<void(int)> *fn;
            {
                std::unique_lock<std::mutex> lk(m_);
                cv_.wait(lk, [&] { return quit_ || epoch_ != seen; });
                if (quit_) {
                    return;
                }
                seen = epoch_;
                n = n_;
                fn = fn_;
            }
            if (fn) {
                drain(seen, n, fn);
            }
        }
    }
    std::vector<std::thread> th_;
    std::mutex m_;
    std::condition_variable cv_, cv_done_;
    const std::function<void(int)> *fn_ = nullptr;
    int n_ = 0;
    std::atomic<unsigned long long> next_{0};
    std::atomic<int> pending_{0};
    unsigned long long epoch_ = 0;
    bool quit_ = false;
};

/* host pictures are staged on the device through a ring of ENC_STAGE_SLOTS buffers: prefetch() may run that many
 * steps minus one ahead of step(), which lets the copy engine work through the long I-picture steps of a GOP and
 * keeps the short P-picture steps fed (H2D of a step's pictures takes longer than a P step's kernels) */
#define ENC_STAGE_SLOTS 4

struct EncLane {
    DSV_ENCODER *enc = nullptr; /* host-side state of this sequence */
    DevFrame pad[2], recon[2], pyr[2][DSV_MAX_PYRAMID_LEVELS], xf, pred;
    DevFrame qrec; /* picture report of an intra-only engine: the reconstruction its pictures otherwise never get */
    int cur = 0, have_ref = 0;
    DevMV *d_mvf[DSV_MAX_PYRAMID_LEVELS + 1] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    int2 *d_aux = nullptr;
    int32_t *coef = nullptr, *llx[3] = {nullptr, nullptr, nullptr}, *dv[3] = {nullptr, nullptr, nullptr};
    uint8_t *tflags = nullptr; /* tile flags of the three planes (sbt.cuh), g.total_tiles bytes */
    uint8_t *hz_dense = nullptr; /* HZCC dense-chunk lists (hzcc.cuh), g.total_chunks * HZ_DENSE_BYTES */
    uint8_t *d_pkt = nullptr, *d_in[ENC_STAGE_SLOTS] = {};
    int in_sel = 0;                 /* staging buffer the next inline copy / prefetch writes */
    const uint8_t *stage_src[ENC_STAGE_SLOTS] = {}; /* host picture on its way into / held by each staging buffer */
    unsigned pkt_dirty = 0;
    size_t pkt_cap = 0; /* bytes allocated at d_pkt */
    uint8_t *h_head = nullptr; /* pinned: packet head assembled on the host */
    /* per-step decisions */
    DSV_FNUM fnum = 0;
    int gop_start = 0, is_ref = 0, has_ref = 0, forced_intra = 0, quant = 0;
    unsigned head_bytes = 0;
};
/* a lane's device buffers (plane_jobs.cpp), for EncEngine and the kernel-level encoder and motion handles alike: inter
 * lanes also get the reference frames, `levels` pyramid levels and the search scratch.  d_mvf[0] and d_in[] point into
 * the owner's lane-major arrays: they are neither allocated nor freed here. */
void enc_lane_alloc(EncLane &l, const CodecGeom &g, bool inter, int levels, size_t pkt_bytes);
void enc_lane_free(EncLane &l);

/* optional destination for a lane's packets: written back to back at `at` instead of into fresh DSV_BUFs */
struct PktSink {
    uint8_t *at;
    size_t room;
    int overflow;
    int mapped; /* destination is mapped pinned host memory: packets leave through an SM copy kernel */
};

/*
 * Single-sequence sharding (long.cpp, dsvb_encode_long): the three phases of a picture run at different times.
 *   analyse  phase 1 only -- ingest, pyramid, luma sum and the motion search against the lane's previous ORIGINAL
 *            picture (source-only data, dsv_encoder.c:231-236): any lane can do it for any picture;
 *   (host)   the serial pass over all pictures in order makes the decisions and writes the packet heads;
 *   code     phase 3 with those decisions given: residual, transform, entropy coding, reconstruction.  Pictures
 *            between two I pictures form a chain; chains are independent and run one per lane.
 */
struct LongAnalysis {
    unsigned long long luma_sum; /* of the smallest pyramid level */
    int nintra;                  /* blocks the search marked intra */
    DevMV *mvs;                  /* nblk vectors of level 0 (host memory) */
};
struct LongPlan {
    int analyse;       /* 1: analysis step (all lanes of a step share the mode) */
    int search;        /* analyse: search against the lane's previous picture (0: the lane's first picture) */
    LongAnalysis *out; /* analyse: results */
    /* code: */
    DSV_FNUM fnum;
    int has_ref, is_ref, quant;
    int forced_intra;      /* an I picture where the GOP asked for a P picture (picture report only) */
    const DevMV *mvs;      /* has_ref: vectors from the analysis pass */
    const uint8_t *stable; /* stable_blocks of this picture (nblk bytes) */
    const uint8_t *head;   /* packet head: header .. quantiser, head_bytes long */
    unsigned head_bytes;
};

/* GOP bookkeeping of one picture (dsv_encoder.c:624-652): host state only */
void gop_bookkeeping(DSV_ENCODER *enc, bool inter, DSV_FNUM fnum, int *gop_start, int *is_ref, int *has_ref);
/* phase 2 of one picture: scene cut / intra share -> frame type, quantiser, stability map, motion side info ->
 * packet head.  top_samples = samples of the smallest pyramid level (the luma average's divisor). */
void decide_and_head(DSV_ENCODER *enc, const CodecGeom &g, bool inter, int top_samples, unsigned long long luma_sum, int nintra,
                     const DevMV *mvs, DSV_FNUM fnum, int is_ref, int *has_ref, int *forced_intra, int *quant, uint8_t *head,
                     unsigned *head_bytes);
static inline size_t head_capacity(const CodecGeom &g) { return 512 + (size_t) g.nblk * 48; }
void make_metadata_packet(DSV_ENCODER *enc, DSV_BUF *buf);

class EncEngine {
public:
    EncEngine(const DSV_META &md, int gop, int pyramid_levels, int lanes);
    ~EncEngine();
    /* encode one picture on each of lane_ids[0..n): src[k] is that lane's input, bufs[k] receives 1 or 2
     * packets (metadata first), nbufs[k] their count.  plan (optional, n entries): see LongPlan. */
    void step(int n, const int *lane_ids, const PicRef *src, DSV_BUF (*bufs)[2], int *nbufs, PktSink *sinks = nullptr,
              const LongPlan *plan = nullptr);
    /* forget a lane's references (a new chain starts on it) */
    void reset_lane(int lane) { lanes_[(size_t) lane].have_ref = 0; }
    /* the next step's kernels start after `ev` (uploads made by the caller on a stream of its own) */
    void wait_event(cudaEvent_t ev)
    {
        if (ev) {
            CUDA_CHECK(cudaStreamWaitEvent(st_, ev, 0));
        }
    }
    /* test hook: the tile flags (sbt.cuh) the lane's last picture left behind, Y then U then V; returns their count */
    int tile_flags(int lane, uint8_t *out, int cap)
    {
        const int n = g_.total_tiles < cap ? g_.total_tiles : cap;
        CUDA_CHECK(cudaMemcpy(out, lanes_[(size_t) lane].tflags, (size_t) n, cudaMemcpyDeviceToHost));
        return g_.total_tiles;
    }
    int pyramid_levels() const { return levels_; }
    bool inter() const { return inter_; }
    /* start copying the NEXT step's host pictures to the device on the copy stream while the current step computes */
    void prefetch(int n, const int *lane_ids, const PicRef *src);
    /* attach a sequence's host state to a lane and forget the lane's references */
    void bind(int lane, DSV_ENCODER *enc)
    {
        lanes_[(size_t) lane].enc = enc;
        lanes_[(size_t) lane].have_ref = 0;
    }
    int lanes() const { return L_; }
    const CodecGeom &geom() const { return g_; }
    EngineStats stats;
    KernelTimes ktimes; /* every launch of step(), by kernel name */
    /* Live timing brackets every launch with two timing events, whose timestamps travel to host memory: cheap on an
     * idle link, but a stream's next operation waits for them, and behind a saturated PCIe direction that adds
     * ~40 us to EVERY launch (measured: device-resident encode 40 -> 81 ms next to an unrelated bulk D2H copy).
     * Off unless asked for (dsvb_*_set_kernel_timing, DSV_KERNEL_TIMES=1). */
    bool time_kernels = false;
    /* Per-picture report (dsvb_enc_set_picture_info): when on, every coding step also measures each picture's squared
     * error against its reconstruction and fills pic_info[k] (pic_info_ok[k] = 0: picture k was dropped, no record).
     * Costs one more launch per step, plus the inverse transform (3 launches) in steps whose pictures are not
     * references.  Off: nothing of it runs or is allocated. */
    bool picture_info = false;
    std::vector<DSVB_PICINFO> pic_info;
    /* SSIM report (dsvb_enc_set_picture_ssim), independent of picture_info: when on, every coding step also measures
     * each plane's SSIM against the reconstruction and fills pic_ssim[k].  One more launch per step, plus the inverse
     * transform as above.  Off: nothing of it runs or is allocated. */
    bool picture_ssim = false;
    std::vector<DSVB_PICSSIM> pic_ssim;
    std::vector<char> pic_info_ok; /* with either report on: picture k of the last step has records (0: dropped) */
    int device = 0;

private:
    void enable_reports(bool sse, bool ssim);
    CodecGeom g_;
    bool inter_;
    int levels_;
    int L_;
    cudaStream_t st_ = 0, st_copy_ = 0;
    cudaEvent_t ev_[7] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t ev_search_ = nullptr; /* vectors and luma sums are on the host */
    cudaEvent_t ev_sizes_ = nullptr;  /* packet sizes are on the host */
    cudaEvent_t ev_pref_[ENC_STAGE_SLOTS] = {}; /* per staging slot: prefetch copies done */
    std::vector<EncLane> lanes_;
    StepArena arena_;
    /* lane-major arrays shared by all lanes so that one copy moves every lane's data */
    DevMV *d_mv0_ = nullptr, *h_mv0_ = nullptr;  /* level-0 motion fields */
    uint8_t *d_stab_ = nullptr, *h_stab_ = nullptr;
    uint8_t *d_misc_ = nullptr, *h_misc_ = nullptr; /* per lane: u64 luma sum, i32 intra count, pad */
    HzChunk *d_chunks_ = nullptr;
    HzFrame *d_frames_ = nullptr, *h_frames_ = nullptr;
    void *h_pk_ = nullptr; /* packet egress copy list (mapped pinned) */
    /* 3 sums per lane of each report, allocated when a step first runs with that report on; h_* mapped pinned */
    unsigned long long *d_sse_ = nullptr, *h_sse_ = nullptr;
    unsigned long long *d_ssim_ = nullptr, *h_ssim_ = nullptr;
    HostPool *pool_ = nullptr;
    uint8_t *d_in_all_[ENC_STAGE_SLOTS] = {}; /* packed-picture staging of all lanes, lane pitch in_pitch_ */
    size_t in_pitch_ = 0;
};

struct DecLane {
    DevFrame out[2];
    int cur = 0, have_ref = 0;
    int32_t *coef = nullptr, *llx[3] = {nullptr, nullptr, nullptr};
    uint8_t *tflags = nullptr; /* tile flags of the three planes (sbt.cuh), g.total_tiles bytes, 16-byte padded */
    HzDecPlaneBufs hz[3];
    uint8_t *d_pkt = nullptr, *h_pkt[2] = {nullptr, nullptr}; /* host staging alternates with the step parity */
    size_t pkt_alloc = 0;
    uint8_t *d_draw = nullptr; /* dense copy of the picture for the debug overlay (lazy) */
    /* per-step */
    int has_ref = 0, is_ref = 0, quant = 0, nplanes = 0, ok = 0, drawn = 0, noout = 0;
    DSV_FNUM fnum = 0;
    HzPlaneData pd[3];
};
/* a lane's device buffers (plane_jobs.cpp), for DecEngine and the kernel-level decoder handle alike; the free also
 * releases the packet staging and overlay copy that DecEngine::step grows on demand */
void dec_lane_alloc(DecLane &l, const CodecGeom &g);
void dec_lane_free(DecLane &l);
/* plane directory of a picture packet (decoder.cpp): from byte `at` of pkt (len bytes) on, up to three planes, each a
 * 32-bit big-endian length and that many bytes.  Fills pd[] with bodies in d_pkt, the device copy of pkt, and returns
 * the number of planes before the first whose length is out of range or which starts past the end. */
int parse_plane_dir(const uint8_t *pkt, unsigned len, unsigned at, const CodecGeom &g, const uint8_t *d_pkt, HzPlaneData pd[3]);

/* one packet of one lane */
struct PktRef {
    const uint8_t *data;     /* host bytes (always needed: the head is parsed on the host) */
    const uint8_t *dev_data; /* optional device copy of the same bytes (skips the H2D copy) */
    unsigned len;
};
struct OutRef {
    uint8_t *plane[3];
    int stride[3];
    int on_device;
};

class DecEngine {
public:
    DecEngine(const DSV_META &md, int lanes);
    ~DecEngine();
    /* decode one PICTURE packet on each of lane_ids[0..n); codes[k] = DSV_DEC_OK / DSV_DEC_ERROR, fnums[k] =
     * frame number; on OK the picture is written to out[k] */
    void step(int n, const int *lane_ids, const PktRef *pkts, const OutRef *out, int *codes, DSV_FNUM *fnums);
    int draw_mode = 0; /* DSV_DECODER.draw_info: overlay painted on the OUTPUT of P pictures (dsv_decoder.c:441-447) */
    /* host-destined pictures leave on the copy stream while the next step computes: wait for all of them */
    void flush();
    const CodecGeom &geom() const { return g_; }
    /* -out420p (dsv_main.c:674-699): pictures leave as 4:2:0 whatever the stream's subsampling; out_geom() is
     * the layout of what step() writes */
    void set_out420(bool on);
    const CodecGeom &out_geom() const { return og_; }
    int lanes() const { return L_; }
    void reset_lane(int lane) { lanes_[(size_t) lane].have_ref = 0; }
    bool matches(const DSV_META &md) const { return md.width == g_.w && md.height == g_.h && md.subsamp == g_.subsamp; }
    EngineStats stats;
    KernelTimes ktimes; /* every launch of step(), by kernel name; read one step late (collect) */
    bool time_kernels = false; /* see EncEngine::time_kernels */
    int device = 0;

private:
    CodecGeom g_, og_;
    int L_;
    int max_nblk_;
    size_t pkt_cap_;
    cudaStream_t st_ = 0, st_copy_ = 0;
    /* a step's host-side inputs (descriptor arena, vectors, stability bits, packet staging) and its timing events
     * exist twice: the host parses step t+1 while the GPU still runs step t */
    cudaEvent_t ev_[2][4] = {{nullptr, nullptr, nullptr, nullptr}, {nullptr, nullptr, nullptr, nullptr}};
    cudaEvent_t ev_end_[2] = {nullptr, nullptr};
    struct Pending {
        bool valid = false, timed = false;
        int pictures = 0, p_pictures = 0;
    } pending_[2];
    void collect(int parity);
    cudaEvent_t ev_done_ = nullptr, ev_copied_[2] = {nullptr, nullptr};
    unsigned long long step_no_ = 0;
    bool prev_nonref_ = false;
    std::vector<DecLane> lanes_;
    StepArena arena_[2];
    DevMV *d_mv_ = nullptr, *h_mv_[2] = {nullptr, nullptr};
    uint8_t *d_stab_ = nullptr, *h_stab_[2] = {nullptr, nullptr};
    uint8_t *d_out_all_[2] = {nullptr, nullptr}; /* packed-picture egress staging of all lanes (step parity) */
    size_t out_pitch_ = 0;
};

static inline double host_now_ms()
{
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6;
}
DSV_FRAME *mk_frame_pinned(int format, int width, int height); /* support.cpp */
bool meta_supported(const DSV_META &m);
void enc_prepare_state(DSV_ENCODER *enc);
void parse_metadata_packet(const uint8_t *pkt, unsigned len, DSV_META *m);

} // namespace dsv
