/*
 * batch_state.h -- what batch.cpp (dsvb_encode / dsvb_decode) and long.cpp (single-sequence and multi-GPU sharding)
 * share: the objects behind the opaque handles and the option-block helpers.
 */
#pragma once
#include <cstring>

#include "dsv1_b200_batch.h"

#include "dsv1_b200.h"

#include "engine.h"

enum {
    CFG_W, CFG_H, CFG_SUBSAMP, CFG_FPS_NUM, CFG_FPS_DEN, CFG_ASPECT_NUM, CFG_ASPECT_DEN,
    CFG_GOP, CFG_QUALITY, CFG_RC_MODE, CFG_BITRATE, CFG_DO_SCD, CFG_SCD_DELTA, CFG_INTRA_PCT,
    CFG_PYR_LEVELS, CFG_STABLE_REFRESH, CFG_MAX_Q_STEP, CFG_MIN_QUALITY, CFG_MAX_QUALITY,
    CFG_MIN_I_QUALITY, CFG_HM_NUDGE, CFG_COUNT
};

struct DSVB_ENC {
    int cfg[CFG_COUNT];
    int lanes, device;
    dsv::EncEngine *eng;
    std::vector<DSV_ENCODER> state;
    /* dsvb_encode_long: pinned packet staging (one slot per lane) and the device-resident picture cache */
    uint8_t *h_stage = nullptr;
    size_t stage_slot = 0;
    uint8_t *d_cache = nullptr;
    size_t cache_bytes = 0;
    cudaStream_t cache_stream = nullptr;
    cudaEvent_t cache_ev[2] = {nullptr, nullptr};
    /* picture report of the last encode call: records per sequence, valid when the report was on and the call succeeded */
    bool info_valid = false;
    std::vector<std::vector<DSVB_PICINFO>> info;
    bool ssim_valid = false; /* SSIM report of the last encode call, the same way */
    std::vector<std::vector<DSVB_PICSSIM>> ssim;
};

struct DSVB_DEC {
    int lanes, device;
    int draw_info = 0, out420 = 0, time_kernels = -1; /* -1: the engine's default (DSV_KERNEL_TIMES) */
    dsv::DecEngine *eng;
    dsv::EngineStats carried; /* stats of engines replaced after a format change */
};

namespace dsv {
void use_device(int device);
int host_mapped(const void *p);
void apply_cfg(DSV_ENCODER *enc, const int *cfg);
void release_state(DSV_ENCODER *enc);
/* one stretch of a container handed to a decoder lane: a whole stream, or one I-delimited chain of a long one */
struct DecSegment {
    const uint8_t *data, *dev; /* host bytes; optional device copy of the same bytes */
    long len;
    int got_meta;              /* the picture format is already known (chains that do not start with metadata) */
    uint8_t *out;              /* pictures land at out + fnum * frame_bytes */
    long out_cap;
    int frames;                /* out: pictures decoded */
};
int decode_segments(DSVB_DEC *d, int nseg, DecSegment *segs, int out_on_device);
/* dsvb_*_picture_info / dsvb_*_picture_ssim: the records of sequence seq, at most cap of them; their count, or -1 */
template <typename R> int copy_records(bool valid, const std::vector<std::vector<R>> &recs, int seq, R *out, int cap)
{
    if (!valid || seq < 0 || seq >= (int) recs.size()) {
        return -1;
    }
    const std::vector<R> &r = recs[(size_t) seq];
    const int n = (int) r.size();
    if (out && cap > 0) {
        memcpy(out, r.data(), sizeof(R) * (size_t) (n < cap ? n : cap));
    }
    return n;
}
} // namespace dsv
