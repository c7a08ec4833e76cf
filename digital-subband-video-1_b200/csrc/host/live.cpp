/*
 * live.cpp -- live streams on the lock-step engines (dsvb_enc_open / _push / _close, dsvb_dec_open / _push / _close):
 * pictures and packets arrive one per stream at a time and every push is one engine step over the streams it lists.
 * A stream is a lane: its DSV_ENCODER runs the reference's host state machine exactly as dsv_enc does (bind() gives
 * it a lane of its own), so a stream's bytes do not depend on which other streams share its steps or when they were
 * opened.  The decoder walks each stream's packet like dsv_dec and decodes the picture packets of a push in one step.
 */
#include "batch_state.h"

using namespace dsv;

/* ids[0..n) are distinct lanes whose state is `want`; nothing is touched otherwise */
static bool live_ids_ok(const std::vector<uint8_t> &live, int n, const int *ids, bool (*want)(uint8_t))
{
    const int L = (int) live.size();
    if (n < 0 || n > L || (n > 0 && !ids)) {
        return false;
    }
    std::vector<char> seen((size_t) L, 0);
    for (int k = 0; k < n; k++) {
        const int id = ids[k];
        if (id < 0 || id >= L || seen[(size_t) id] || !want(live[(size_t) id])) {
            return false;
        }
        seen[(size_t) id] = 1;
    }
    return true;
}

static int live_take_lane(std::vector<uint8_t> &live, int *count)
{
    for (size_t i = 0; i < live.size(); i++) {
        if (live[i] == LIVE_FREE) {
            live[i] = LIVE_OPEN;
            ++*count;
            return (int) i;
        }
    }
    return -1;
}

/* ---- encoder ---------------------------------------------------------------------------------- */

extern "C" int dsvb_enc_open(DSVB_ENC *e)
{
    DSV_API_BEGIN
    use_device(e->device);
    const int id = live_take_lane(e->live, &e->live_open);
    if (id < 0) {
        return -1;
    }
    /* a fresh encoder from the object's options, as dsvb_encode starts each sequence */
    DSV_ENCODER *enc = &e->state[(size_t) id];
    apply_cfg(enc, e->cfg);
    enc_prepare_state(enc);
    e->eng->bind(id, enc);
    return id;
    DSV_API_END(-100)
}

extern "C" long dsvb_enc_push_bound(DSVB_ENC *e)
{
    return (long) (64 + enc_packet_cap(e->eng->geom())); /* metadata packet (make_metadata_packet: <= 64 bytes) + picture */
}

extern "C" int dsvb_enc_push(DSVB_ENC *e, int n, const int *ids, const uint8_t *const *pics, int on_device,
                             uint8_t *const *out, const long *caps, long *lens)
{
    DSV_API_BEGIN
    if (!live_ids_ok(e->live, n, ids, [](uint8_t s) { return s == LIVE_OPEN; })) {
        return -2;
    }
    if (n == 0) {
        return 0;
    }
    use_device(e->device);
    const CodecGeom &g = e->eng->geom();
    const bool report = e->eng->picture_info, report_ssim = e->eng->picture_ssim;
    e->info_valid = e->ssim_valid = false;
    std::vector<PicRef> src((size_t) n);
    std::vector<PktSink> sinks((size_t) n);
    std::vector<int> nb((size_t) n);
    std::vector<DSV_BUF> bufs((size_t) 2 * n);
    for (int k = 0; k < n; k++) {
        for (int p = 0; p < 3; p++) {
            src[(size_t) k].plane[p] = pics[k] + g.plane_off[p];
            src[(size_t) k].stride[p] = g.pw[p];
        }
        src[(size_t) k].on_device = on_device;
        const bool room = out[k] && caps[k] > 0;
        sinks[(size_t) k].at = out[k];
        sinks[(size_t) k].room = room ? (size_t) caps[k] : 0;
        sinks[(size_t) k].overflow = 0;
        sinks[(size_t) k].mapped = room ? host_mapped(out[k]) : 0;
    }
    /* the step ends in a stream synchronisation: every packet is in its sink when it returns */
    e->eng->step(n, ids, src.data(), reinterpret_cast<DSV_BUF(*)[2]>(bufs.data()), nb.data(), sinks.data());
    int rc = 0;
    e->info.assign(report ? (size_t) n : 0, std::vector<DSVB_PICINFO>());
    e->ssim.assign(report_ssim ? (size_t) n : 0, std::vector<DSVB_PICSSIM>());
    for (int k = 0; k < n; k++) {
        const PktSink &sk = sinks[(size_t) k];
        if (sk.overflow) {
            /* the encoder state has moved past bytes the caller does not hold: the stream cannot continue */
            lens[k] = -1;
            e->live[(size_t) ids[k]] = LIVE_BROKEN;
            rc = -1;
            continue;
        }
        lens[k] = (long) (sk.at - out[k]);
        if (e->eng->pic_info_ok.size() > (size_t) k && e->eng->pic_info_ok[(size_t) k]) {
            if (report) {
                e->info[(size_t) k].push_back(e->eng->pic_info[(size_t) k]);
            }
            if (report_ssim) {
                e->ssim[(size_t) k].push_back(e->eng->pic_ssim[(size_t) k]);
            }
        }
    }
    e->info_valid = report;
    e->ssim_valid = report_ssim;
    return rc;
    DSV_API_END(-100)
}

extern "C" int dsvb_enc_close(DSVB_ENC *e, int id, uint8_t *out, long cap, long *len)
{
    DSV_API_BEGIN
    if (id < 0 || id >= e->lanes || e->live[(size_t) id] == LIVE_FREE) {
        return -2;
    }
    DSV_ENCODER *enc = &e->state[(size_t) id];
    DSV_BUF eos[1];
    dsv_enc_end_of_stream(enc, eos);
    const bool fits = out && cap >= (long) eos[0].len;
    if (fits) {
        memcpy(out, eos[0].data, eos[0].len);
    }
    if (len) {
        *len = fits ? (long) eos[0].len : -1;
    }
    dsv_buf_free(&eos[0]);
    release_state(enc);
    e->live[(size_t) id] = LIVE_FREE;
    e->live_open--;
    return fits ? 0 : -1;
    DSV_API_END(-100)
}

/* ---- decoder ---------------------------------------------------------------------------------- */

extern "C" int dsvb_dec_open(DSVB_DEC *d)
{
    const int id = live_take_lane(d->live, &d->live_open);
    if (id >= 0 && d->eng) {
        d->eng->reset_lane(id);
    }
    return id;
}

extern "C" void dsvb_dec_close(DSVB_DEC *d, int id)
{
    if (id >= 0 && id < d->lanes && d->live[(size_t) id] != LIVE_FREE) {
        d->live[(size_t) id] = LIVE_FREE;
        d->live_open--;
    }
}

extern "C" int dsvb_dec_push(DSVB_DEC *d, int n, const int *ids, const uint8_t *const *pkts, const uint8_t *const *pkts_dev,
                             const long *lens, uint8_t *const *out, int out_on_device, int *codes, long long *fnums)
{
    DSV_API_BEGIN
    if (!live_ids_ok(d->live, n, ids, [](uint8_t s) { return s != LIVE_FREE; })) {
        return -2;
    }
    use_device(d->device);
    /* host-only packets first (dsv_decoder.c:300-331); picture packets of streams with a known format go to one step */
    std::vector<int> lane((size_t) n), slot((size_t) n), step_codes((size_t) n);
    std::vector<PktRef> pk((size_t) n);
    std::vector<OutRef> outs((size_t) n);
    std::vector<DSV_FNUM> fn((size_t) n);
    int m = 0;
    for (int k = 0; k < n; k++) {
        const int id = ids[k];
        const uint8_t *hdr = pkts[k];
        const long len = lens[k];
        codes[k] = DSV_DEC_ERROR;
        fnums[k] = -1;
        if (!hdr || len < DSV_PACKET_HDR_SIZE || hdr[0] != DSV_FOURCC_0 || hdr[1] != DSV_FOURCC_1 || hdr[2] != DSV_FOURCC_2 ||
            hdr[3] != DSV_FOURCC_3) {
            continue;
        }
        const int type = hdr[DSV_PACKET_TYPE_OFFSET];
        if (type == DSV_PT_META) {
            DSV_META md;
            memset(&md, 0, sizeof(md));
            parse_metadata_packet(hdr, (unsigned) len, &md);
            if (!meta_supported(md)) {
                continue;
            }
            if (d->eng && !d->eng->matches(md)) {
                /* one picture format per object: it may change only while no other stream depends on it */
                bool held = false;
                for (int i = 0; i < d->lanes && !held; i++) {
                    held = i != id && d->live[(size_t) i] == LIVE_HAS_META;
                }
                if (held) {
                    continue;
                }
            }
            dec_use_format(d, md);
            d->live[(size_t) id] = LIVE_HAS_META;
            codes[k] = DSV_DEC_GOT_META;
            continue;
        }
        if (type == DSV_PT_EOS) {
            codes[k] = DSV_DEC_EOS;
            continue;
        }
        if (!DSV_PT_IS_PIC(type)) {
            continue;
        }
        if (d->live[(size_t) id] != LIVE_HAS_META) {
            codes[k] = DSV_DEC_OK; /* a picture before any metadata is skipped (dsv_decoder.c:327-331) */
            continue;
        }
        const CodecGeom &og = d->eng->out_geom();
        lane[(size_t) m] = id;
        slot[(size_t) m] = k;
        pk[(size_t) m].data = hdr;
        pk[(size_t) m].dev_data = pkts_dev ? pkts_dev[k] : nullptr;
        pk[(size_t) m].len = (unsigned) len;
        for (int p = 0; p < 3; p++) {
            outs[(size_t) m].plane[p] = out && out[k] ? out[k] + og.plane_off[p] : nullptr;
            outs[(size_t) m].stride[p] = og.pw[p];
        }
        outs[(size_t) m].on_device = out_on_device;
        m++;
    }
    if (m > 0) {
        d->eng->step(m, lane.data(), pk.data(), outs.data(), step_codes.data(), fn.data());
        d->eng->flush(); /* the pictures are complete in out[] when the call returns */
        for (int q = 0; q < m; q++) {
            codes[slot[(size_t) q]] = step_codes[(size_t) q];
            fnums[slot[(size_t) q]] = fn[(size_t) q] == (DSV_FNUM) -1 ? -1 : (long long) fn[(size_t) q];
        }
    }
    return 0;
    DSV_API_END(-100)
}
