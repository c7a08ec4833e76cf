/*
 * batch.cpp -- dsvb_*: the additive throughput API (include/dsv1_b200_batch.h) on top of the lock-step
 * engines.  Sequences are taken in waves of `lanes`; inside a wave picture t of every lane is one engine
 * step.  Streams come out exactly as the per-picture API emits them (metadata at every GOP start, link
 * fields, EOS), because every lane runs the same host-side state machine (a DSV_ENCODER per lane).
 */
#include "batch_state.h"

#include "bits.h"

using namespace dsv;

namespace dsv {
void synth_launch(int w, int h, int hs, int vs, int start, int n, int seed, int cut, uint8_t *d_out, cudaStream_t st);
}

namespace dsv {

void use_device(int device) { CUDA_CHECK(cudaSetDevice(device)); }

/* pinned (cudaMallocHost / cudaHostRegister) host memory is addressable by kernels under UVA */
int host_mapped(const void *p)
{
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return a.type == cudaMemoryTypeHost;
}

void apply_cfg(DSV_ENCODER *enc, const int *cfg)
{
    DSV_META md;
    memset(&md, 0, sizeof(md));
    md.width = cfg[CFG_W];
    md.height = cfg[CFG_H];
    md.subsamp = cfg[CFG_SUBSAMP];
    md.fps_num = cfg[CFG_FPS_NUM];
    md.fps_den = cfg[CFG_FPS_DEN];
    md.aspect_num = cfg[CFG_ASPECT_NUM];
    md.aspect_den = cfg[CFG_ASPECT_DEN];
    dsv_enc_init(enc);
    dsv_enc_set_metadata(enc, &md);
    enc->gop = cfg[CFG_GOP];
    enc->scene_change_delta = cfg[CFG_SCD_DELTA];
    enc->do_scd = cfg[CFG_DO_SCD];
    enc->intra_pct_thresh = cfg[CFG_INTRA_PCT];
    enc->quality = cfg[CFG_QUALITY];
    enc->rc_mode = cfg[CFG_RC_MODE];
    enc->bitrate = (unsigned) cfg[CFG_BITRATE];
    enc->max_q_step = cfg[CFG_MAX_Q_STEP];
    enc->min_quality = cfg[CFG_MIN_QUALITY];
    enc->max_quality = cfg[CFG_MAX_QUALITY];
    enc->min_I_frame_quality = cfg[CFG_MIN_I_QUALITY];
    enc->rc_high_motion_nudge = cfg[CFG_HM_NUDGE];
    enc->pyramid_levels = cfg[CFG_PYR_LEVELS];
    enc->stable_refresh = (unsigned) cfg[CFG_STABLE_REFRESH];
    dsv_enc_start(enc);
}

void release_state(DSV_ENCODER *enc)
{
    if (enc->stability) {
        dsv_free(enc->stability);
        enc->stability = NULL;
    }
    if (enc->stable_blocks) {
        dsv_free(enc->stable_blocks);
        enc->stable_blocks = NULL;
    }
}

} // namespace dsv

static void fill_stats(const EngineStats &s, int device, int lanes, double *out)
{
    out[0] = s.sbt_fwd_ms;
    out[1] = (double) s.sbt_fwd_launches;
    out[2] = (double) s.sbt_fwd_bytes;
    out[3] = s.sbt_inv_ms;
    out[4] = (double) s.sbt_inv_launches;
    out[5] = (double) s.sbt_inv_bytes;
    out[6] = (double) s.kernel_launches;
    out[7] = (double) s.h2d_bytes;
    out[8] = (double) s.d2h_bytes;
    out[9] = (double) s.pictures;
    out[10] = (double) device;
    out[11] = (double) lanes;
    out[12] = s.host_ms;
    out[13] = s.bmc_ms;
    out[14] = (double) s.bmc_launches;
    out[15] = (double) s.bmc_bytes;
}

extern "C" DSVB_ENC *dsvb_enc_create(const int *cfg, int lanes, int device)
{
    DSV_API_BEGIN
    if (lanes < 1 || lanes > 1024) {
        return nullptr;
    }
    use_device(device);
    DSVB_ENC *e = new DSVB_ENC();
    memcpy(e->cfg, cfg, sizeof(e->cfg));
    e->lanes = lanes;
    e->device = device;
    e->state.resize((size_t) lanes);
    e->live.assign((size_t) lanes, LIVE_FREE);
    /* one probe state fixes the block grid and the pyramid depth for the engine */
    DSV_ENCODER probe;
    apply_cfg(&probe, cfg);
    enc_prepare_state(&probe);
    e->eng = new EncEngine(probe.vidmeta, probe.gop, probe.pyramid_levels, lanes);
    release_state(&probe);
    return e;
    DSV_API_END(nullptr)
}

extern "C" void dsvb_enc_destroy(DSVB_ENC *e)
{
    if (e) {
        use_device(e->device);
        for (int i = 0; i < e->lanes; i++) {
            if (e->live[(size_t) i] != LIVE_FREE) { /* live streams never closed */
                release_state(&e->state[(size_t) i]);
            }
        }
        delete e->eng;
        cudaFreeHost(e->h_stage);
        cudaFree(e->d_cache);
        if (e->cache_stream) {
            cudaStreamDestroy(e->cache_stream);
            cudaEventDestroy(e->cache_ev[0]);
            cudaEventDestroy(e->cache_ev[1]);
        }
        delete e;
    }
}

extern "C" void dsvb_enc_stats(DSVB_ENC *e, double *stats, int reset)
{
    fill_stats(e->eng->stats, e->device, e->lanes, stats);
    if (reset) {
        e->eng->stats = EngineStats();
    }
}

static void fill_ktimes(KernelTimes *kt, double *ms, double *launches, int reset)
{
    const int n = kt_count();
    for (int i = 0; i < n; i++) {
        ms[i] = kt ? kt->ms[i] : 0.0;
        launches[i] = kt ? (double) kt->launches[i] : 0.0;
    }
    if (kt && reset) {
        kt->reset();
    }
}

extern "C" int dsvb_enc_tile_flags(DSVB_ENC *e, int lane, uint8_t *out, int cap)
{
    DSV_API_BEGIN
    use_device(e->device);
    if (lane < 0 || lane >= e->lanes) {
        return -1;
    }
    return e->eng->tile_flags(lane, out, cap);
    DSV_API_END(-100)
}

extern "C" void dsvb_enc_set_kernel_timing(DSVB_ENC *e, int on) { e->eng->time_kernels = on != 0; }
extern "C" void dsvb_dec_set_kernel_timing(DSVB_DEC *d, int on)
{
    d->time_kernels = on != 0;
    if (d->eng) {
        d->eng->time_kernels = on != 0;
    }
}

extern "C" void dsvb_enc_set_picture_info(DSVB_ENC *e, int on) { e->eng->picture_info = on != 0; }
extern "C" void dsvb_enc_set_picture_ssim(DSVB_ENC *e, int on) { e->eng->picture_ssim = on != 0; }

extern "C" int dsvb_enc_picture_info(DSVB_ENC *e, int seq, DSVB_PICINFO *out, int cap)
{
    return copy_records(e->info_valid, e->info, seq, out, cap);
}

extern "C" int dsvb_enc_picture_ssim(DSVB_ENC *e, int seq, DSVB_PICSSIM *out, int cap)
{
    return copy_records(e->ssim_valid, e->ssim, seq, out, cap);
}

extern "C" int dsvb_kernel_count(void) { return kt_count(); }
extern "C" const char *dsvb_kernel_name(int i) { return kt_name(i); }
extern "C" void dsvb_enc_kernel_times(DSVB_ENC *e, double *ms, double *launches, int reset)
{
    fill_ktimes(&e->eng->ktimes, ms, launches, reset);
}

extern "C" int dsvb_encode(DSVB_ENC *e, int nseq, int nframes, const uint8_t *const *yuv, int on_device,
                           uint8_t *const *streams, const long *caps, long *lens)
{
    DSV_API_BEGIN
    if (e->live_open) {
        return -2; /* the waves rebind lanes 0..n-1: open live streams hold some of them */
    }
    use_device(e->device);
    const CodecGeom &g = e->eng->geom();
    const int L = e->lanes;
    int rc = 0;
    const bool report = e->eng->picture_info, report_ssim = e->eng->picture_ssim;
    e->info_valid = e->ssim_valid = false;
    e->info.assign(report ? (size_t) nseq : 0, std::vector<DSVB_PICINFO>());
    e->ssim.assign(report_ssim ? (size_t) nseq : 0, std::vector<DSVB_PICSSIM>());
    std::vector<int> ids((size_t) L);
    std::vector<PicRef> src((size_t) L), next((size_t) L);
    std::vector<PktSink> sinks((size_t) L);
    std::vector<int> nb((size_t) L);
    std::vector<DSV_BUF> bufs((size_t) 2 * L);
    for (int base = 0; base < nseq; base += L) {
        const int n = nseq - base < L ? nseq - base : L;
        for (int k = 0; k < n; k++) {
            apply_cfg(&e->state[(size_t) k], e->cfg);
            enc_prepare_state(&e->state[(size_t) k]);
            e->eng->bind(k, &e->state[(size_t) k]);
            ids[(size_t) k] = k;
            sinks[(size_t) k].at = streams[base + k];
            sinks[(size_t) k].room = (size_t) caps[base + k];
            sinks[(size_t) k].overflow = 0;
            sinks[(size_t) k].mapped = host_mapped(streams[base + k]);
        }
        auto pictures = [&](int t, std::vector<PicRef> &dst) {
            for (int k = 0; k < n; k++) {
                const uint8_t *f = yuv[base + k] + (size_t) t * g.frame_bytes;
                for (int p = 0; p < 3; p++) {
                    dst[(size_t) k].plane[p] = f + g.plane_off[p];
                    dst[(size_t) k].stride[p] = g.pw[p];
                }
                dst[(size_t) k].on_device = on_device;
            }
        };
        /* host pictures cross PCIe on the copy stream up to ENC_STAGE_SLOTS - 1 steps ahead of the encoder: the copy
         * engine keeps working through the long I-picture step and the short P-picture steps never wait for input */
        const int ahead = ENC_STAGE_SLOTS - 1;
        for (int t = 0; !on_device && t < ahead && t < nframes; t++) {
            pictures(t, next);
            e->eng->prefetch(n, ids.data(), next.data());
        }
        for (int t = 0; t < nframes; t++) {
            if (!on_device && t + ahead < nframes) {
                pictures(t + ahead, next);
                e->eng->prefetch(n, ids.data(), next.data());
            }
            pictures(t, src);
            e->eng->step(n, ids.data(), src.data(), reinterpret_cast<DSV_BUF(*)[2]>(bufs.data()), nb.data(), sinks.data());
            for (int k = 0; (report || report_ssim) && k < n; k++) {
                if (e->eng->pic_info_ok[(size_t) k] && report) {
                    e->info[(size_t) (base + k)].push_back(e->eng->pic_info[(size_t) k]);
                }
                if (e->eng->pic_info_ok[(size_t) k] && report_ssim) {
                    e->ssim[(size_t) (base + k)].push_back(e->eng->pic_ssim[(size_t) k]);
                }
            }
        }
        for (int k = 0; k < n; k++) {
            PktSink &sk = sinks[(size_t) k];
            DSV_BUF eos[1];
            dsv_enc_end_of_stream(&e->state[(size_t) k], eos);
            if (!sk.overflow && sk.room >= eos[0].len) {
                memcpy(sk.at, eos[0].data, eos[0].len);
                sk.at += eos[0].len;
                sk.room -= eos[0].len;
            } else {
                sk.overflow = 1;
            }
            dsv_buf_free(&eos[0]);
            lens[base + k] = sk.overflow ? -1 : (long) (sk.at - streams[base + k]);
            if (sk.overflow) {
                rc = -1;
            }
            release_state(&e->state[(size_t) k]);
        }
    }
    e->info_valid = report && rc == 0;
    e->ssim_valid = report_ssim && rc == 0;
    return rc;
    DSV_API_END(-100)
}

extern "C" DSVB_DEC *dsvb_dec_create(int lanes, int device)
{
    if (lanes < 1 || lanes > 1024) {
        return nullptr;
    }
    DSVB_DEC *d = new DSVB_DEC();
    d->lanes = lanes;
    d->device = device;
    d->eng = nullptr;
    d->live.assign((size_t) lanes, LIVE_FREE);
    return d;
}

extern "C" void dsvb_dec_destroy(DSVB_DEC *d)
{
    if (d) {
        use_device(d->device);
        delete d->eng;
        delete d;
    }
}

static void add_stats(EngineStats &a, const EngineStats &b)
{
    a.sbt_fwd_ms += b.sbt_fwd_ms;
    a.sbt_inv_ms += b.sbt_inv_ms;
    a.sbt_fwd_launches += b.sbt_fwd_launches;
    a.sbt_inv_launches += b.sbt_inv_launches;
    a.sbt_fwd_bytes += b.sbt_fwd_bytes;
    a.sbt_inv_bytes += b.sbt_inv_bytes;
    a.kernel_launches += b.kernel_launches;
    a.h2d_bytes += b.h2d_bytes;
    a.d2h_bytes += b.d2h_bytes;
    a.pictures += b.pictures;
    a.host_ms += b.host_ms;
    a.bmc_ms += b.bmc_ms;
    a.bmc_launches += b.bmc_launches;
    a.bmc_bytes += b.bmc_bytes;
}

extern "C" void dsvb_dec_set_draw_info(DSVB_DEC *d, int mode)
{
    d->draw_info = mode;
    if (d->eng) {
        d->eng->draw_mode = mode;
    }
}

extern "C" void dsvb_dec_set_out420p(DSVB_DEC *d, int on)
{
    d->out420 = on;
    if (d->eng) {
        d->eng->set_out420(on != 0);
    }
}

extern "C" void dsvb_dec_kernel_times(DSVB_DEC *d, double *ms, double *launches, int reset)
{
    fill_ktimes(d->eng ? &d->eng->ktimes : nullptr, ms, launches, reset);
}

extern "C" void dsvb_dec_stats(DSVB_DEC *d, double *stats, int reset)
{
    EngineStats s = d->carried;
    if (d->eng) {
        add_stats(s, d->eng->stats);
    }
    fill_stats(s, d->device, d->lanes, stats);
    if (reset) {
        d->carried = EngineStats();
        if (d->eng) {
            d->eng->stats = EngineStats();
        }
    }
}

static unsigned be32(const uint8_t *p) { return ((unsigned) p[0] << 24) | ((unsigned) p[1] << 16) | ((unsigned) p[2] << 8) | p[3]; }

void dsv::dec_use_format(DSVB_DEC *d, const DSV_META &md)
{
    if (d->eng && !d->eng->matches(md)) {
        add_stats(d->carried, d->eng->stats);
        delete d->eng;
        d->eng = nullptr;
    }
    if (!d->eng) {
        d->eng = new DecEngine(md, d->lanes);
        if (d->time_kernels >= 0) {
            d->eng->time_kernels = d->time_kernels != 0;
        }
        d->eng->draw_mode = d->draw_info;
        d->eng->set_out420(d->out420 != 0);
    }
}

/*
 * Lock-step decode of a set of container segments: every lane walks its segment packet by packet (metadata / EOS
 * are host-only), picture packets of all lanes are one engine step; a lane that finishes its segment takes the
 * next one from the queue, so ragged segment lengths do not leave lanes idle.
 */
int dsv::decode_segments(DSVB_DEC *d, int nseg, DecSegment *segs, int out_on_device)
{
    const int L = d->lanes;
    int rc = 0;
    std::vector<long> pos((size_t) L);
    std::vector<int> cur((size_t) L, -1), got_meta((size_t) L);
    std::vector<int> ids((size_t) L), seg_of((size_t) L), codes((size_t) L);
    std::vector<PktRef> pk((size_t) L);
    std::vector<OutRef> outs((size_t) L);
    std::vector<DSV_FNUM> fn((size_t) L);
    int next_seg = 0;
    bool stepped = false; /* the engine (= the picture format) can only be replaced before the first step of a call */
    for (int s = 0; s < nseg; s++) {
        segs[s].frames = 0;
    }
    for (;;) {
        /* advance every lane to its next picture packet */
        int m = 0;
        for (int k = 0; k < L; k++) {
            for (;;) {
                if (cur[(size_t) k] < 0) {
                    if (next_seg >= nseg) {
                        break;
                    }
                    cur[(size_t) k] = next_seg++;
                    pos[(size_t) k] = 0;
                    got_meta[(size_t) k] = segs[cur[(size_t) k]].got_meta;
                    if (d->eng) {
                        d->eng->reset_lane(k);
                    }
                }
                DecSegment &sg = segs[cur[(size_t) k]];
                const long at = pos[(size_t) k];
                if (at + DSV_PACKET_HDR_SIZE > sg.len) {
                    cur[(size_t) k] = -1;
                    continue;
                }
                const uint8_t *hdr = sg.data + at;
                if (hdr[0] != DSV_FOURCC_0 || hdr[1] != DSV_FOURCC_1 || hdr[2] != DSV_FOURCC_2 || hdr[3] != DSV_FOURCC_3) {
                    cur[(size_t) k] = -1;
                    rc = -4;
                    continue;
                }
                long size = (long) be32(hdr + DSV_PACKET_NEXT_OFFSET);
                if (size == 0) {
                    size = DSV_PACKET_HDR_SIZE;
                }
                if (size < DSV_PACKET_HDR_SIZE || at + size > sg.len) {
                    cur[(size_t) k] = -1;
                    rc = -3;
                    continue;
                }
                const int type = hdr[DSV_PACKET_TYPE_OFFSET];
                pos[(size_t) k] = at + size;
                if (type == DSV_PT_META) {
                    DSV_META md;
                    memset(&md, 0, sizeof(md));
                    parse_metadata_packet(hdr, (unsigned) size, &md);
                    if (!meta_supported(md)) {
                        cur[(size_t) k] = -1;
                        rc = -5;
                        continue;
                    }
                    if (d->eng && !d->eng->matches(md) && (stepped || m > 0)) {
                        cur[(size_t) k] = -1; /* one picture format per call */
                        rc = -6;
                        continue;
                    }
                    dec_use_format(d, md);
                    got_meta[(size_t) k] = 1;
                    continue;
                }
                if (type == DSV_PT_EOS) {
                    cur[(size_t) k] = -1;
                    continue;
                }
                if (!DSV_PT_IS_PIC(type) || !got_meta[(size_t) k] || !d->eng) {
                    continue; /* pictures before metadata are skipped (dsv_decoder.c:327-331) */
                }
                ids[(size_t) m] = k;
                seg_of[(size_t) m] = cur[(size_t) k];
                pk[(size_t) m].data = hdr;
                pk[(size_t) m].dev_data = sg.dev ? sg.dev + at : nullptr;
                pk[(size_t) m].len = (unsigned) size;
                /* frame number decides where the picture lands: peek it (fnum follows the header) */
                const CodecGeom &g = d->eng->out_geom();
                const DSV_FNUM fno = be32(hdr + DSV_PACKET_HDR_SIZE);
                const size_t off = (size_t) fno * g.frame_bytes;
                if (off + g.frame_bytes > (size_t) sg.out_cap) {
                    /* no room: decode (references must stay in step) into the lane's own frame only */
                    for (int p = 0; p < 3; p++) {
                        outs[(size_t) m].plane[p] = nullptr;
                    }
                } else {
                    for (int p = 0; p < 3; p++) {
                        outs[(size_t) m].plane[p] = sg.out + off + g.plane_off[p];
                        outs[(size_t) m].stride[p] = g.pw[p];
                    }
                }
                outs[(size_t) m].on_device = out_on_device;
                m++;
                break;
            }
        }
        if (m == 0) {
            break;
        }
        d->eng->step(m, ids.data(), pk.data(), outs.data(), codes.data(), fn.data());
        stepped = true;
        for (int q = 0; q < m; q++) {
            if (codes[(size_t) q] == DSV_DEC_OK && outs[(size_t) q].plane[0]) {
                segs[seg_of[(size_t) q]].frames++;
            }
        }
    }
    if (d->eng) {
        d->eng->flush(); /* the last pictures are still leaving on the copy stream */
    }
    return rc;
}

extern "C" int dsvb_decode(DSVB_DEC *d, int nseq, const uint8_t *const *streams, const uint8_t *const *streams_dev,
                           const long *lens, uint8_t *const *out, const long *out_caps, int out_on_device, int *frames)
{
    DSV_API_BEGIN
    if (d->live_open) {
        return -2; /* the segments would take over lanes that open live streams hold */
    }
    use_device(d->device);
    std::vector<DecSegment> segs((size_t) nseq);
    for (int s = 0; s < nseq; s++) {
        segs[(size_t) s] = DecSegment{streams[s], streams_dev ? streams_dev[s] : nullptr, lens[s], 0, out[s], out_caps[s], 0};
    }
    const int rc = decode_segments(d, nseq, segs.data(), out_on_device);
    for (int s = 0; s < nseq; s++) {
        frames[s] = segs[(size_t) s].frames;
    }
    return rc;
    DSV_API_END(-100)
}

extern "C" void *dsvb_host_alloc(size_t bytes)
{
    DSV_API_BEGIN
    void *p = nullptr;
    if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) {
        return nullptr;
    }
    return p;
    DSV_API_END(nullptr)
}

extern "C" void dsvb_host_free(void *p) { cudaFreeHost(p); }

extern "C" int dsvb_synth_device(int w, int h, int subsamp, int start, int n, int seed, int cut, uint8_t *d_out, int device)
{
    DSV_API_BEGIN
    use_device(device);
    synth_launch(w, h, (subsamp >> 2) & 3, subsamp & 3, start, n, seed, cut, d_out, 0);
    CUDA_CHECK(cudaDeviceSynchronize());
    return 0;
    DSV_API_END(-100)
}
