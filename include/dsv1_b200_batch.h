/*
 * dsv1_b200_batch.h -- additive throughput API of libdsv1_b200.so (not in the reference).
 *
 * The reference API (dsv_enc / dsv_dec, dsv_encoder.h:112-121, dsv_decoder.h:52-59) is synchronous and
 * one-picture-at-a-time.  Independent sequences (closed GOPs, whole clips) have no data dependence on
 * each other, so this API runs up to `lanes` of them in LOCK STEP on one GPU: picture t of every lane goes
 * through each pipeline stage in one batched kernel launch.  The bytes produced for a sequence are exactly
 * the bytes the per-picture API produces for it (same code path with one lane); tests/test_gpu_batch.py
 * checks that.  One object per GPU and host thread; objects on different GPUs are independent (no
 * collective: segments are gathered in order on the host, SURVEY.md section 8e).
 *
 * cfg is the 21-int option block of tools/api_harness.c (the fields dsv_main.c:463-489 sets on
 * DSV_ENCODER / DSV_META): w h subsamp fps_num fps_den aspect_num aspect_den gop quality rc_mode bitrate
 * do_scd scd_delta intra_pct pyr_levels stable_refresh max_q_step min_quality max_quality min_i_quality hm_nudge
 */
#ifndef DSV1_B200_BATCH_H
#define DSV1_B200_BATCH_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct DSVB_ENC DSVB_ENC;
typedef struct DSVB_DEC DSVB_DEC;

#define DSVB_NSTATS 16
/* stats[]: 0 sbt_fwd_ms 1 sbt_fwd_launches 2 sbt_fwd_bytes 3 sbt_inv_ms 4 sbt_inv_launches 5 sbt_inv_bytes
 *          6 kernel_launches 7 h2d_bytes 8 d2h_bytes 9 pictures 10 device 11 lanes 12 host_ms
 *          13 bmc_ms 14 bmc_launches 15 bmc_bytes */

DSVB_ENC *dsvb_enc_create(const int *cfg, int lanes, int device);
void dsvb_enc_destroy(DSVB_ENC *e);
/*
 * Encode nseq sequences of nframes pictures each.  yuv[s]: packed planar pictures of sequence s back to
 * back, in host memory (on_device = 0; pinned memory avoids a staging copy) or device memory (1).
 * streams[s] (host, caps[s] bytes) receives the complete .dsv stream (META, PIC..., EOS) of sequence s,
 * lens[s] its length.  Returns 0, or -1 if a stream buffer is too small.
 */
int dsvb_encode(DSVB_ENC *e, int nseq, int nframes, const uint8_t *const *yuv, int on_device,
                uint8_t *const *streams, const long *caps, long *lens);
void dsvb_enc_stats(DSVB_ENC *e, double *stats, int reset);
/* Test hook: the per-tile band flags (one byte per 128x64 tile, planes Y, U, V back to back; bit 0 = the tile's
 * level-1 band blocks hold a non-zero coefficient, bit 1 = its level-2 blocks do) that the last picture coded on
 * `lane` left behind.  Returns the number of tiles per picture, at most `cap` bytes are written. */
int dsvb_enc_tile_flags(DSVB_ENC *e, int lane, uint8_t *out, int cap);

DSVB_DEC *dsvb_dec_create(int lanes, int device);
void dsvb_dec_destroy(DSVB_DEC *d);
/*
 * Decode nseq .dsv streams of one picture format.  streams[s]/lens[s]: host bytes (always required: packet
 * heads are parsed on the host).  streams_dev (optional, may be NULL): device copies of the same bytes;
 * when given no packet is copied host->device.  out[s]: packed planar pictures at offset
 * fnum * frame_bytes, in host (out_on_device = 0) or device (1) memory of out_caps[s] bytes.
 * frames[s] receives the number of pictures decoded.  Returns 0, or a negative value on a malformed container.
 */
int dsvb_decode(DSVB_DEC *d, int nseq, const uint8_t *const *streams, const uint8_t *const *streams_dev,
                const long *lens, uint8_t *const *out, const long *out_caps, int out_on_device, int *frames);
void dsvb_dec_stats(DSVB_DEC *d, double *stats, int reset);
/* DSV_DECODER.draw_info for the streams decoded from now on (DSV_DRAW_* bits, dsv_decoder.h:38-41): the debug
 * overlay is painted on the pictures written to `out`, never on the decoder's own references */
void dsvb_dec_set_draw_info(DSVB_DEC *d, int mode);
/* the CLI's -out420p (dsv_main.c:674-699, util.c:54-93): when on, pictures of 4:4:4 / 4:2:2 / 4:1:1 streams are
 * written to `out` as packed 4:2:0 (frame size w*h + 2*ceil(w/2)*ceil(h/2)), converted on the device */
void dsvb_dec_set_out420p(DSVB_DEC *d, int on);

/*
 * ONE long sequence sharded over the lanes of a GPU (csrc/host/long.cpp).  Pictures between two I pictures
 * (periodic GOP starts AND forced ones: scene cuts, too many intra blocks) form a chain; chains are independent
 * once the serial per-picture decisions are made, so they run one per lane.  Three phases: (A) pyramid + motion
 * search of every picture against its ORIGINAL predecessor, batched over the lanes (source-only data,
 * dsv_encoder.c:231-236); (B) one serial host pass in picture order for frame types, the stability tracker
 * (dsv_encoder.c:329-408) and the packet heads; (C) residual / transform / entropy coding / reconstruction of
 * the chains; then an ordered gather with metadata packets, frame numbers and prev/next links
 * (dsv_encoder.c:170-192,427-461) exactly as dsv_enc writes them: the stream is byte-identical to feeding the
 * pictures to dsv_enc one by one.  ABR streams (rc_mode != CRF) serialise on packet sizes and run on one lane.
 * yuv: nframes packed planar pictures (host, or device when on_device = 1).  info (optional, 4 ints):
 * chains, forced I pictures, longest chain, GPUs used (0: single-GPU entry, 1: serial ABR path).
 * Returns 0, -1 if `stream` (cap bytes) is too small, -100 on a CUDA failure.
 */
int dsvb_encode_long(DSVB_ENC *e, int nframes, const uint8_t *yuv, int on_device, uint8_t *stream, long cap, long *len,
                     int *info);
/* One container decoded with its chains (cut at every picture that has no reference, dsv_decoder.c:286-472)
 * spread over the lanes.  stream_dev (optional): device copy of the same bytes.  Pictures land at
 * out + fnum * frame_bytes like dsvb_decode. */
int dsvb_decode_long(DSVB_DEC *d, const uint8_t *stream, const uint8_t *stream_dev, long len, uint8_t *out, long out_cap,
                     int out_on_device, int *frames);

/*
 * Several GPUs of one box behind one object: one engine and one host thread per GPU, no collective (SURVEY.md
 * section 8e: replicas + ordered host gather).  devices: ndev CUDA ordinals (NULL: 0..ndev-1); cfg may be NULL
 * for a decode-only object.  All buffers are host memory (pinned memory avoids staging copies).
 *   dsvb_multi_encode / _decode        whole sequences / streams dealt to the GPUs in contiguous runs
 *   dsvb_multi_encode_long             one sequence: phase A over contiguous runs of pictures, phase B on the
 *                                      calling thread, phase C over contiguous runs of chains, ordered gather
 *   dsvb_multi_decode_long             one container cut at GOP starts into one run of chains per GPU
 */
typedef struct DSVB_MULTI DSVB_MULTI;
DSVB_MULTI *dsvb_multi_create(const int *cfg, int lanes, int ndev, const int *devices);
void dsvb_multi_destroy(DSVB_MULTI *m);
int dsvb_multi_encode(DSVB_MULTI *m, int nseq, int nframes, const uint8_t *const *yuv, uint8_t *const *streams,
                      const long *caps, long *lens);
int dsvb_multi_decode(DSVB_MULTI *m, int nseq, const uint8_t *const *streams, const long *lens, uint8_t *const *out,
                      const long *out_caps, int *frames);
int dsvb_multi_encode_long(DSVB_MULTI *m, int nframes, const uint8_t *yuv, uint8_t *stream, long cap, long *len, int *info);
int dsvb_multi_decode_long(DSVB_MULTI *m, const uint8_t *stream, long len, uint8_t *out, long out_cap, int *frames);

/* Live per-kernel timing: every kernel launch of an engine step is bracketed by CUDA events on the engine's stream.
 * dsvb_kernel_count() names are registered so far (at most 64, in order of first launch); ms[i] / launches[i]
 * (arrays of at least 64 doubles) receive the accumulated device time and launch count of kernel i since the last
 * reset.  The decoder reads a step's events when the step has left the GPU (dsvb_decode returns after that). */
/* Timing is OFF by default (or DSV_KERNEL_TIMES=1 in the environment): the two timing events per launch cost ~40 us
 * per launch when a PCIe direction is saturated by picture traffic, because their timestamps go to host memory.
 * The sbt / bmc entries of the stats block are filled only while timing is on. */
void dsvb_enc_set_kernel_timing(DSVB_ENC *e, int on);
void dsvb_dec_set_kernel_timing(DSVB_DEC *d, int on);
int dsvb_kernel_count(void);
const char *dsvb_kernel_name(int i);
void dsvb_enc_kernel_times(DSVB_ENC *e, double *ms, double *launches, int reset);
void dsvb_dec_kernel_times(DSVB_DEC *d, double *ms, double *launches, int reset);

/*
 * Per-picture report of the encoders: squared error against the source, frame type, quantiser and size of every
 * coded picture.  Off by default; while off the encoders do exactly what they do without it (same bytes, launches
 * and allocations).  When on, the closed-loop reconstruction (what a decoder outputs) is compared with the source on
 * the GPU, and pictures that are not references (every picture of a gop = 0 encoder) get the inverse transform they
 * otherwise skip.  The streams do not change.
 *   dsvb_enc_picture_info / dsvb_multi_picture_info: the records of sequence `seq` of the last dsvb_encode /
 *   dsvb_multi_encode call (seq 0 for dsvb_encode_long / dsvb_multi_encode_long), in picture order.  Returns the
 *   number of records and writes at most `cap` of them; -1 if the report was off during that call, the call failed,
 *   or seq is out of range.
 * PSNR of plane p: 10 * log10(255^2 * samples[p] / sse[p]) (infinite when sse[p] == 0).
 */
typedef struct DSVB_PICINFO { /* 72 bytes, no padding */
    uint64_t sse[3];          /* sum over the plane of (source - reconstruction)^2, Y U V; the reconstruction is what a decoder outputs */
    int64_t samples[3];       /* pw * ph per plane, so PSNR = 10 log10(255^2 * samples / sse) needs no subsampling rules */
    int64_t fnum;             /* frame number written in the packet */
    int32_t is_p;             /* 1: P picture, 0: I picture */
    int32_t forced_intra;     /* a P picture turned into I (scene change / intra share) */
    int32_t quant;            /* quantiser written in the packet */
    int32_t bytes;            /* picture packet incl. head; metadata packets excluded */
} DSVB_PICINFO;
void dsvb_enc_set_picture_info(DSVB_ENC *e, int on);
int dsvb_enc_picture_info(DSVB_ENC *e, int seq, DSVB_PICINFO *out, int cap);
void dsvb_multi_set_picture_info(DSVB_MULTI *m, int on);
int dsvb_multi_picture_info(DSVB_MULTI *m, int seq, DSVB_PICINFO *out, int cap);

/*
 * SSIM report of the encoders: the SSIM of every plane of every coded picture against the source, measured on the GPU
 * on the same closed-loop reconstruction as the report above.  Independent of it: either can be on without the other.
 * Off by default; while off the encoders do exactly what they do without it.  When on it costs one kernel per step,
 * and pictures that are not references get the inverse transform they otherwise skip.  The streams do not change.
 *   dsvb_enc_picture_ssim / dsvb_multi_picture_ssim: as dsvb_enc_picture_info / dsvb_multi_picture_info (records of
 *   sequence `seq` of the last encode call in picture order, at most `cap` written, the count returned; -1 if the
 *   SSIM report was off during that call, the call failed, or seq is out of range).
 * Definition (x264 / ffmpeg, 8-bit), for a plane of pw x ph samples, source a, reconstruction b:
 *   4x4 blocks: bw = pw / 4, bh = ph / 4 (the last pw % 4 columns and ph % 4 rows are not read);
 *   windows: the 2x2 groups of blocks at block positions (i, j), 0 <= i < bw - 1, 0 <= j < bh - 1 (8x8 samples,
 *   stride 4); per window, over its 64 samples in int64: s1 = sum a, s2 = sum b, ss = sum (a^2 + b^2), s12 = sum ab,
 *   vars = 64 ss - s1^2 - s2^2, covar = 64 s12 - s1 s2,
 *   ssim_w = (double) ((2 s1 s2 + 416) (2 covar + 235963)) / (double) ((s1^2 + s2^2 + 416) (vars + 235963))
 *   (IEEE round to nearest); the plane's sum S = sum over windows of rint(ssim_w * 2^32) (ties to even), in int64,
 *   and ssim = (double) S / 2^32 / windows.  The sum of integers makes the result independent of summation order,
 *   lanes and devices.
 * dB form: -10 * log10(1 - ssim) (infinite when ssim == 1).
 */
typedef struct DSVB_PICSSIM { /* 48 bytes, no padding */
    double ssim[3];           /* mean SSIM over the plane's 8x8 windows (stride 4), Y U V; NaN when windows[p] == 0 */
    int64_t windows[3];       /* (pw/4 - 1) * (ph/4 - 1), 0 when a plane has fewer than 8 samples in either direction */
} DSVB_PICSSIM;
void dsvb_enc_set_picture_ssim(DSVB_ENC *e, int on);
int dsvb_enc_picture_ssim(DSVB_ENC *e, int seq, DSVB_PICSSIM *out, int cap);
void dsvb_multi_set_picture_ssim(DSVB_MULTI *m, int on);
int dsvb_multi_picture_ssim(DSVB_MULTI *m, int seq, DSVB_PICSSIM *out, int cap);

/* pinned host memory for inputs / outputs of the calls above */
void *dsvb_host_alloc(size_t bytes);
void dsvb_host_free(void *p);

/* SURVEY.md Appendix-C synthetic content, generated on the GPU straight into DEVICE memory (bench / test
 * utility; bit-identical to oracle/synth.c): n pictures starting at index `start`, packed planar */
int dsvb_synth_device(int w, int h, int subsamp, int start, int n, int seed, int cut, uint8_t *d_out, int device);

#ifdef __cplusplus
}
#endif
#endif /* DSV1_B200_BATCH_H */
