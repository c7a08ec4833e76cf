/*
 * dsv1_b200_kernels.h -- kernel-level C ABI of libdsv1_b200.so (HOST buffers in, HOST buffers out).
 *
 * One entry point per hot-path subsystem of the reference (dsv_internal.h:94-109, dsv_encoder.h:132),
 * with flat pointer+size signatures so that a test, a benchmark or a foreign-language binding can
 * drive a single subsystem.  Every call copies its inputs to the GPU, runs the CUDA kernels and
 * copies the result back; there is no host implementation behind any of these symbols.
 * The same signatures are implemented by the checker libraries (oracle/ref_harness.c: ref_*,
 * oracle/dsv1_port.c: port_*) -- those are test infrastructure, never linked into this library.
 *
 * Return value: 0 (or a byte/element count where stated) on success, negative on bad arguments.
 */
#ifndef DSV1_B200_KERNELS_H
#define DSV1_B200_KERNELS_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* dsv_fwd_sbt (sbt.c:630-651): pix = ph rows of `stride` bytes with >= cw valid columns;
 * coef_out = cw*ch int32, dense.  cw, ch even and >= 16. */
int dsvk_fwd_sbt(const uint8_t *pix, int stride, int pw, int ph, int cw, int ch, int isP, int32_t *coef_out);

/* dsv_inv_sbt (sbt.c:653-714): c = plane index (0 = luma: smoothing-filtered inverse), q = frame quant. */
int dsvk_inv_sbt(int32_t *coef_io, int cw, int ch, int q, int isP, int c, uint8_t *pix_out, int stride, int pw, int ph);

/* dsv_fwd_sbt followed by the quantise + in-place dequantise half of hzcc_enc (hzcc.c:156-281), fused
 * as the encoder runs it.  dv_out (optional) receives the first-visit symbols of positions hzcc scans
 * twice; returns their count. */
int dsvk_fwd_sbt_q(const uint8_t *pix, int stride, int pw, int ph, int cw, int ch, int isP, int c, int q,
                   const uint8_t *stable, int nbh, int nbv, int32_t *coef_out, int32_t *dv_out);

/* dsv_encode_plane (hzcc.c:449-476): raw coefficients in, plane bytes (plen field first) out,
 * coef_io <- dequantised.  Returns the number of bytes written. */
int dsvk_encode_plane(int32_t *coef_io, int cw, int ch, int q, int isP, int c, const uint8_t *stable,
                      int nbh, int nbv, uint8_t *out, int out_cap);

/* dsv_decode_plane (hzcc.c:478-496): `in` points just after the 32-bit plen field. */
int dsvk_decode_plane(const uint8_t *in, int plen, int cw, int ch, int q, int isP, int c,
                      const uint8_t *stable, int nbh, int nbv, int32_t *coef_out);

/* mk_pyramid (dsv_encoder.c:194-217): luma pyramid levels 1..levels of a packed planar frame, packed
 * one after another into out; out_w/out_h receive each level's size. */
int dsvk_pyramid(const uint8_t *yuv, int w, int h, int subsamp, int levels, uint8_t *out, int *out_w, int *out_h);

/* dsv_hme (hme.c:730-741) on two packed planar ORIGINAL frames; mv_out = nbh*nbv DSV_MV records
 * (12 bytes each, dsv.h:137-150).  Returns the intra-block percentage. */
int dsvk_hme(const uint8_t *src_yuv, const uint8_t *ref_yuv, int w, int h, int subsamp, int blk_w, int blk_h,
             int levels, void *mv_out);

/* dsv_sub_pred (bmc.c:318-331): pred_out = prediction, resid_out = clamp(inp - pred + 128). */
int dsvk_sub_pred(const void *mvs, int w, int h, int subsamp, int blk_w, int blk_h, const uint8_t *inp_yuv,
                  const uint8_t *ref_yuv, uint8_t *pred_out, uint8_t *resid_out);

/* dsv_add_pred (bmc.c:333-346): out = clamp(pred + resid - 128). */
int dsvk_add_pred(const void *mvs, int w, int h, int subsamp, int blk_w, int blk_h, const uint8_t *resid_yuv,
                  const uint8_t *ref_yuv, uint8_t *out_yuv);

/* ---- batch entry points: the transform and entropy-coding kernels configured as the engines launch them ----------
 * One call is one launch sequence over n pictures x 3 planes, with the engines' own job filling: tile flags, the
 * encoder's list scratch and dense pack pass, the fused prediction add, the multi-picture job mapping.  Frames are
 * packed planar (w x h luma, then two chroma planes of the subsampled size); coefficient planes are the three
 * planes' dense coefficients back to back (chroma sizes rounded up to even); tile flags are one byte per 128x64 tile
 * of each plane, planes back to back (bit 0: level-1 band blocks hold a non-zero, bit 1: level-2). */
typedef struct DSVK_PIC {
    int isP;               /* P picture (inter quantiser tables; the encoder adds the prediction in its inverse) */
    int quant;             /* frame quantiser */
    const uint8_t *stable; /* encoder, decoder: nbh * nbv stability bytes of the handle's block grid */
    unsigned start_byte;   /* encoder: length of the packet head, plane 0 starts here */
    unsigned cap;          /* encoder: packet bytes the coder may use, <= dsvk_enc_pkt_bytes() */
} DSVK_PIC;

/* encoder lanes for up to max_pics pictures of one format; each lane keeps its packet buffer (only the dirty prefix
 * is cleared before the next call), list scratch and tile flags from call to call */
void *dsvk_enc_create(int w, int h, int subsamp, int blk_w, int blk_h, int max_pics);
long dsvk_enc_pkt_bytes(void *enc);
void dsvk_enc_destroy(void *enc);
/* forward transform + quantiser -> HZCC scan / prefix / pack -> inverse (+ prediction) of pictures 0..n-1 in lanes
 * 0..n-1.  in: n frames (the picture, or its residual for P); pred: n frames or NULL.  Out, per picture k:
 * pkt_out[k * (dsvk_enc_pkt_bytes() + 4096)...] the whole packet buffer including a 4096-byte guard past the largest
 * cap; info_out[8k..8k+7] = overflow, total bytes, plane bytes Y/U/V, dv counts Y/U/V; coef_out = the dequantised
 * coefficients; dv_out[(3k + p) * dv_pitch...] the plane's double-visit side buffer, dv_pitch = 2 * (w + h) + 16;
 * tflags_out = the flags the forward kernel wrote; recon_out = the reconstruction. */
int dsvk_enc_run(void *enc, int n, const DSVK_PIC *pics, const uint8_t *in, const uint8_t *pred, uint8_t *pkt_out,
                 unsigned *info_out, int32_t *coef_out, int32_t *dv_out, uint8_t *tflags_out, uint8_t *recon_out);

/* the entropy-coding half of dsvk_enc_run on caller coefficients (coef_io: raw in, dequantised out) and caller tile
 * flags (NULL: no chunk is skipped): quantiser, then scan / prefix / pack with the engine's list scratch (I pictures:
 * sparse and dense lists, P: sparse lists).  pkt_out, info_out and dv_out as for dsvk_enc_run; the packet buffer per
 * picture is enc_packet_cap of the format (dsvk_enc_pkt_bytes of a handle of that format) + 4096 bytes. */
int dsvk_hz_enc_batch(int w, int h, int subsamp, int blk_w, int blk_h, int n, const DSVK_PIC *pics, int32_t *coef_io,
                      const uint8_t *tflags, uint8_t *pkt_out, unsigned *info_out, int32_t *dv_out);

/* inverse transform of n pictures in one launch, geo[3k..3k+2] = w, h, subsamp of picture k (formats may differ).
 * coef: the pictures' coefficient planes back to back; tflags: their tile flags back to back, or NULL (no skipping);
 * pred: n frames, added on the way out to the P pictures (as the engines do), or NULL. */
int dsvk_inv_batch(int n, const int *geo, const DSVK_PIC *pics, const int32_t *coef, const uint8_t *tflags,
                   const uint8_t *pred, uint8_t *out);

/* squared error of n picture pairs in one launch, as the batch encoder's picture report measures it: geo as for
 * dsvk_inv_batch; src / rec hold n packed frames each.  Both are placed in bordered device frames whose border and
 * padding bytes are set to border_fill[0] (src) and border_fill[1] (rec).  sse_out: 3 sums per picture, Y U V. */
int dsvk_sse_batch(int n, const int *geo, const uint8_t *src, const uint8_t *rec, const uint8_t *border_fill, uint64_t *sse_out);
/* SSIM of n picture pairs in one launch, as the batch encoders' SSIM report measures it: geo / src / rec / border_fill
 * as for dsvk_sse_batch.  sum_out: 3 per picture, Y U V = sum over the plane's windows of rint(ssim_w * 2^32) (the
 * definition is at DSVB_PICSSIM, dsv1_b200_batch.h); windows_out: 3 per picture.  -1: a geometry is illegal. */
int dsvk_ssim_batch(int n, const int *geo, const uint8_t *src, const uint8_t *rec, const uint8_t *border_fill,
                    int64_t *sum_out, int64_t *windows_out);

/* decoder lane: coefficient planes and tile flags carry over from one picture to the next */
void *dsvk_dec_create(int w, int h, int subsamp, int blk_w, int blk_h);
void dsvk_dec_destroy(void *dec);
/* entropy decoding of one picture: planes = the three plane records (32-bit big-endian plen, then plen bytes) back to
 * back.  Returns the number of planes decoded; coef_out / tflags_out receive the lane's planes and flags. */
int dsvk_dec_run(void *dec, const DSVK_PIC *pic, const uint8_t *planes, int len, int32_t *coef_out, uint8_t *tflags_out);

/* ---- batch entry points: the motion kernels configured as the engines launch them ----------------------------------
 * The encoder's phase 1 (ingest with border, luma pyramid, luma sum, hierarchical search) and its motion compensation,
 * and the decoder's compensation, with the engines' own descriptor filling and launch order over n lanes.  Frames are
 * packed planar as above; motion fields are nbh * nbv DSV_MV records (12 bytes) per lane, lanes back to back. */
typedef struct DSVK_ME_PIC {
    const uint8_t *src;    /* the packed picture, at any byte address */
    int src_on_device;     /* 1: src is device memory, ingested where it lies; 0: host memory, copied first */
    unsigned stage_offset; /* host src: byte offset (0..255) in the lane's staging buffer it is copied to */
    int has_ref;           /* search against the lane's previous picture, then compensate from its reconstruction */
    int do_sum;            /* luma sum of the smallest pyramid level (scene-change detection) */
    const uint8_t *recon;  /* NULL, or this picture's packed reconstruction: stored and bordered as the encoder's
                              phase 3 stores it, it is the reference of the lane's next compensation */
} DSVK_ME_PIC;

/* lanes for up to max_pics pictures of one format and block grid, with `levels` (1..5) pyramid levels; each lane keeps
 * its ingested frames, pyramids and reconstructions in two buffers that alternate from call to call */
void *dsvk_me_create(int w, int h, int subsamp, int blk_w, int blk_h, int levels, int max_pics);
void dsvk_me_destroy(void *me);
/* bytes of a lane's device allocation of pyramid level `level` (0: the ingested frame), guard bands included */
long dsvk_me_frame_bytes(void *me, int level);
/* pictures 0..n-1 on lanes 0..n-1.  mvs NULL: ingest -> pyramid -> zero -> luma sum -> search -> compensation; mvs =
 * n fields (the long encode's code pass): ingest, then the compensation with those vectors.  Out, per picture k:
 * frames_out = the whole allocation of the ingested frame, then of pyramid levels 1..levels (dsvk_me_frame_bytes);
 * misc_out[2k], [2k+1] = the lane's luma sum and intra-block count; mv_out = the level-0 field; pred_out / resid_out
 * = prediction and residual (has_ref pictures).  -1: bad arguments, or a has_ref picture on a lane without a picture. */
int dsvk_me_run(void *me, int n, const DSVK_ME_PIC *pics, const void *mvs, uint8_t *frames_out, int64_t *misc_out, void *mv_out,
                uint8_t *pred_out, uint8_t *resid_out);
/* the decoder's compensation of n lanes in one launch: out[k] = resid[k] + prediction from ref[k] - 128 with lane k's
 * field (mvs + k * nbh * nbv) where isP[k], resid[k] unchanged otherwise */
int dsvk_add_pred_batch(int w, int h, int subsamp, int blk_w, int blk_h, int n, const int *isP, const void *mvs, const uint8_t *resid,
                        const uint8_t *ref, uint8_t *out);

#ifdef __cplusplus
}
#endif
#endif /* DSV1_B200_KERNELS_H */
