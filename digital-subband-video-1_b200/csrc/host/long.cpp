/*
 * long.cpp -- ONE long sequence sharded over the lanes of a GPU and over several GPUs (dsvb_encode_long,
 * dsvb_decode_long, dsvb_multi_*): the "independent closed GOPs sharded across the GPUs, segments gathered in
 * order on the host" of the project brief, made exact.
 *
 * Re-encoding every GOP with a fresh encoder is NOT byte-identical to the reference: the stability accumulators
 * and their refresh counter run across GOP boundaries (dsv_encoder.c:345-352,812-814), forced I pictures (scene
 * cuts, dsv_encoder.c:538-554; too many intra blocks, dsv_encoder.c:246-253) split a GOP without restarting it, and
 * the previous-picture links (dsv_encoder.c:170-192) chain the packets.  What IS independent:
 *
 *   phase A  per picture t: pyramid, luma average, motion search of t against the ORIGINAL picture t-1
 *            (dsv_encoder.c:231-236): source-only.  Pictures are dealt to the lanes in contiguous runs; a lane
 *            first ingests the picture before its run (no search), then searches picture after picture.
 *   phase B  one serial host pass in picture order over a few kB per picture: GOP bookkeeping, scene cut,
 *            intra share -> frame type; stability tracker; quantiser; the complete packet head (header, frame
 *            number, stability map, motion sub-streams, quantiser).  Same functions as the per-picture API.
 *   phase C  pictures between two I pictures form a chain (closed: an I picture needs no reference); chains run
 *            one per lane, a lane takes the next chain when its own ends.  Residual, transform, entropy coding,
 *            reconstruction = phase 3 of the ordinary engine step with the decisions handed in.
 *   gather   packets are concatenated in picture order; metadata packets go in front of every GOP start
 *            (prev link 0, dsv_encoder.c:427-461), each picture's prev link is the length of the previous
 *            picture packet, EOS closes the stream (dsv_encoder.c:765-778).
 *
 * ABR (rc_mode != CRF) serialises on packet sizes (dsv_encoder.c:84-160,816-848): such sequences run on one
 * lane of one GPU, exactly like dsv_enc.  Several GPUs: one host thread and one engine per GPU, phase A over
 * contiguous runs of pictures, phase B on the calling thread, phase C over contiguous runs of chains; no
 * collective anywhere.  The decoder shards at every picture without a reference (dsv_decoder.c:286-472).
 */
#include "batch_state.h"

#include "bits.h"

#include <thread>

using namespace dsv;

namespace {

unsigned rd_be32(const uint8_t *p) { return ((unsigned) p[0] << 24) | ((unsigned) p[1] << 16) | ((unsigned) p[2] << 8) | p[3]; }
void wr_be32(uint8_t *p, unsigned v)
{
    p[0] = (uint8_t) (v >> 24);
    p[1] = (uint8_t) (v >> 16);
    p[2] = (uint8_t) (v >> 8);
    p[3] = (uint8_t) v;
}

/* everything the phases of one long encode share; the per-device workers only touch disjoint picture ranges */
struct LongCtx {
    const int *cfg = nullptr;
    int nframes = 0;
    const uint8_t *yuv = nullptr;
    int on_device = 0;
    CodecGeom g;
    bool inter = false;
    int levels = 0;
    size_t head_cap = 0;
    std::vector<LongAnalysis> ana;
    std::vector<DevMV> mvs;        /* nframes x nblk */
    std::vector<uint8_t> heads;    /* nframes x head_cap */
    std::vector<uint8_t> stab;     /* nframes x nblk */
    std::vector<LongPlan> plan;
    std::vector<char> gop_start;
    std::vector<int> chain_first;  /* first picture of every chain, plus nframes as the sentinel */
    std::vector<std::vector<uint8_t>> pkt; /* coded picture packets */
    std::vector<DSVB_PICINFO> info;         /* picture report, by picture index */
    std::vector<DSVB_PICSSIM> ssim;         /* SSIM report, by picture index */
    int forced = 0;
    int err = 0;
};

void ctx_init(LongCtx &c, const DSVB_ENC *e, int nframes, const uint8_t *yuv, int on_device)
{
    c.cfg = e->cfg;
    c.nframes = nframes;
    c.yuv = yuv;
    c.on_device = on_device;
    c.g = e->eng->geom();
    c.inter = e->eng->inter();
    c.levels = e->eng->pyramid_levels();
    c.head_cap = head_capacity(c.g);
    const size_t n = (size_t) nframes;
    c.ana.assign(n, LongAnalysis{0, 0, nullptr});
    c.mvs.assign(n * (size_t) c.g.nblk, DevMV());
    for (size_t t = 0; t < n; t++) {
        c.ana[t].mvs = c.mvs.data() + t * (size_t) c.g.nblk;
    }
    c.heads.assign(n * c.head_cap, 0);
    c.stab.assign(n * (size_t) c.g.nblk, 0);
    c.plan.assign(n, LongPlan());
    c.gop_start.assign(n, 0);
    c.pkt.resize(n);
    c.info.assign(e->eng->picture_info ? n : 0, DSVB_PICINFO());
    c.ssim.assign(e->eng->picture_ssim ? n : 0, DSVB_PICSSIM());
}

/*
 * Where picture t is read from.  Host pictures go through a device-resident cache of the whole sequence when it
 * fits (DSV_LONG_CACHE_MB, default 16 GiB): a picture is uploaded when a step first needs it, one step ahead of
 * that step on a copy stream of its own, and both passes then read device memory -- every picture crosses PCIe
 * once.  When the sequence does not fit the passes stream from the host through the engine's own prefetch and
 * every picture crosses twice.
 */
struct PicSource {
    const LongCtx *c = nullptr;
    DSVB_ENC *e = nullptr;
    uint8_t *d_cache = nullptr;
    std::vector<char> resident;
    int parity = 0;

    void open(DSVB_ENC *enc, const LongCtx *ctx)
    {
        c = ctx;
        e = enc;
        d_cache = nullptr;
        if (c->on_device) {
            return;
        }
        size_t budget = (size_t) 16384 << 20;
        if (const char *s = getenv("DSV_LONG_CACHE_MB")) {
            budget = (size_t) atol(s) << 20;
        }
        const size_t need = (size_t) c->nframes * c->g.frame_bytes;
        if (need > budget) {
            return;
        }
        if (e->cache_bytes < need) {
            cudaFree(e->d_cache);
            e->d_cache = nullptr;
            e->cache_bytes = 0;
            if (cudaMalloc(&e->d_cache, need) != cudaSuccess) {
                cudaGetLastError();
                e->d_cache = nullptr;
                return;
            }
            e->cache_bytes = need;
        }
        if (!e->cache_stream) {
            CUDA_CHECK(cudaStreamCreateWithFlags(&e->cache_stream, cudaStreamNonBlocking));
            CUDA_CHECK(cudaEventCreateWithFlags(&e->cache_ev[0], cudaEventDisableTiming));
            CUDA_CHECK(cudaEventCreateWithFlags(&e->cache_ev[1], cudaEventDisableTiming));
        }
        d_cache = e->d_cache;
        resident.assign((size_t) c->nframes, 0);
    }
    bool streams_from_host() const { return !c->on_device && !d_cache; }
    PicRef at(int t) const
    {
        PicRef r;
        const uint8_t *f = (d_cache ? d_cache : c->yuv) + (size_t) t * c->g.frame_bytes;
        for (int p = 0; p < 3; p++) {
            r.plane[p] = f + c->g.plane_off[p];
            r.stride[p] = c->g.pw[p];
        }
        r.on_device = d_cache ? 1 : c->on_device;
        return r;
    }
    /* start the uploads a coming step needs; returns the event that step has to wait for (NULL: nothing) */
    cudaEvent_t upload(const int *frames, int n)
    {
        if (!d_cache) {
            return nullptr;
        }
        const size_t fb = c->g.frame_bytes;
        for (int q = 0; q < n; q++) {
            const int t = frames[q];
            if (!resident[(size_t) t]) {
                CUDA_CHECK(cudaMemcpyAsync(d_cache + (size_t) t * fb, c->yuv + (size_t) t * fb, fb, cudaMemcpyHostToDevice, e->cache_stream));
                resident[(size_t) t] = 1;
                e->eng->stats.h2d_bytes += fb;
            }
        }
        parity ^= 1;
        CUDA_CHECK(cudaEventRecord(e->cache_ev[parity], e->cache_stream));
        return e->cache_ev[parity];
    }
};

/* phase A on one engine: pictures [t0, t1) */
void long_analyse(DSVB_ENC *e, LongCtx &c, PicSource &ps, int t0, int t1)
{
    if (!c.inter || t1 <= t0) {
        return;
    }
    EncEngine *eng = e->eng;
    const int L = e->lanes;
    const int total = t1 - t0;
    const int nl = total < L ? total : L;
    /* lane i owns the run [a_i, b_i); it starts one picture early (its first search reference) unless a_i == 0 */
    std::vector<int> a((size_t) nl), b((size_t) nl), at((size_t) nl);
    for (int i = 0; i < nl; i++) {
        a[(size_t) i] = t0 + (int) ((long long) total * i / nl);
        b[(size_t) i] = t0 + (int) ((long long) total * (i + 1) / nl);
        at[(size_t) i] = a[(size_t) i] > 0 ? a[(size_t) i] - 1 : 0;
        eng->reset_lane(i);
    }
    std::vector<int> ids((size_t) nl), nb((size_t) nl);
    std::vector<PicRef> src((size_t) nl), nxt((size_t) nl);
    std::vector<LongPlan> plan((size_t) nl);
    std::vector<DSV_BUF> bufs((size_t) 2 * nl);
    std::vector<int> fr((size_t) nl);
    auto collect = [&](std::vector<PicRef> &dst, std::vector<int> &lane, const std::vector<int> &pos) {
        int m = 0;
        for (int i = 0; i < nl; i++) {
            if (pos[(size_t) i] < b[(size_t) i]) {
                lane[(size_t) m] = i;
                fr[(size_t) m] = pos[(size_t) i];
                dst[(size_t) m] = ps.at(pos[(size_t) i]);
                m++;
            }
        }
        return m;
    };
    const bool stream_in = ps.streams_from_host();
    std::vector<int> nids((size_t) nl);
    int m = collect(src, ids, at);
    if (stream_in && m) {
        eng->prefetch(m, ids.data(), src.data());
    }
    cudaEvent_t ready = ps.upload(fr.data(), m);
    while (m > 0) {
        for (int q = 0; q < m; q++) {
            const int i = ids[(size_t) q], t = at[(size_t) i];
            LongPlan &p = plan[(size_t) q];
            memset(&p, 0, sizeof(p));
            p.analyse = 1;
            p.search = t >= a[(size_t) i] && t > 0; /* the picture before the run is only ingested */
            p.out = t >= a[(size_t) i] ? &c.ana[(size_t) t] : nullptr;
            p.fnum = (DSV_FNUM) t;
        }
        std::vector<int> after = at;
        for (int q = 0; q < m; q++) {
            after[(size_t) ids[(size_t) q]]++;
        }
        const int m_next = collect(nxt, nids, after);
        if (stream_in && m_next) {
            eng->prefetch(m_next, nids.data(), nxt.data());
        }
        eng->wait_event(ready);
        ready = ps.upload(fr.data(), m_next);
        eng->step(m, ids.data(), src.data(), reinterpret_cast<DSV_BUF(*)[2]>(bufs.data()), nb.data(), nullptr, plan.data());
        at = after;
        m = m_next;
        ids.swap(nids);
        src.swap(nxt);
    }
}

/* phase B: the serial pass (the calling thread, no GPU work) */
void long_decide(LongCtx &c)
{
    DSV_ENCODER enc;
    apply_cfg(&enc, c.cfg);
    enc_prepare_state(&enc);
    const CodecGeom &g = c.g;
    const int top_samples = c.inter ? ceil_shift(g.w, c.levels) * ceil_shift(g.h, c.levels) : 1;
    c.chain_first.clear();
    for (int t = 0; t < c.nframes; t++) {
        const DSV_FNUM fnum = enc.next_fnum++;
        int gop_start, is_ref, has_ref, forced = 0, quant = 0;
        gop_bookkeeping(&enc, c.inter, fnum, &gop_start, &is_ref, &has_ref);
        uint8_t *head = c.heads.data() + (size_t) t * c.head_cap;
        unsigned head_bytes = 0;
        const LongAnalysis &an = c.ana[(size_t) t];
        decide_and_head(&enc, g, c.inter, top_samples, an.luma_sum, an.nintra, an.mvs, fnum, is_ref, &has_ref, &forced, &quant, head,
                        &head_bytes);
        memcpy(c.stab.data() + (size_t) t * g.nblk, enc.stable_blocks, (size_t) g.nblk);
        if (has_ref) {
            enc.refresh_ctr++; /* dsv_encoder.c:812-814 */
        }
        LongPlan &p = c.plan[(size_t) t];
        memset(&p, 0, sizeof(p));
        p.fnum = fnum;
        p.has_ref = has_ref;
        p.is_ref = is_ref;
        p.quant = quant;
        p.forced_intra = (c.inter && !has_ref && !gop_start) ? 1 : 0;
        p.mvs = an.mvs;
        p.stable = c.stab.data() + (size_t) t * g.nblk;
        p.head = head;
        p.head_bytes = head_bytes;
        c.gop_start[(size_t) t] = (char) gop_start;
        c.forced += p.forced_intra; /* I pictures that are not GOP starts */
        if (!has_ref) {
            c.chain_first.push_back(t);
        }
    }
    c.chain_first.push_back(c.nframes);
    release_state(&enc);
}

/* phase C on one engine: chains [k0, k1), one per lane, a lane takes the next chain when its own ends */
void long_code(DSVB_ENC *e, LongCtx &c, PicSource &ps, int k0, int k1)
{
    if (k1 <= k0) {
        return;
    }
    EncEngine *eng = e->eng;
    const int L = e->lanes;
    const CodecGeom &g = c.g;
    if (!e->h_stage) { /* a picture packet per lane, sized like the reference's own packet buffer (dsv_encoder.c:472-491) */
        size_t ub = (size_t) g.w * g.h;
        ub *= (g.subsamp == DSV_SUBSAMP_444) ? 6 : (g.subsamp == DSV_SUBSAMP_422) ? 4 : 2;
        e->stage_slot = (ub + 4096 + (size_t) g.nblk * 48 + 255) & ~(size_t) 255;
        CUDA_CHECK(cudaMallocHost(&e->h_stage, e->stage_slot * (size_t) L));
    }
    std::vector<int> at((size_t) L, -1), end((size_t) L, -1); /* next picture / end of the lane's chain */
    int next_chain = k0;
    std::vector<int> ids((size_t) L), nids((size_t) L), nb((size_t) L), pic((size_t) L), npic((size_t) L);
    std::vector<PicRef> src((size_t) L), nxt((size_t) L);
    std::vector<LongPlan> plan((size_t) L);
    std::vector<PktSink> sinks((size_t) L);
    std::vector<DSV_BUF> bufs((size_t) 2 * L);
    const bool stream_in = ps.streams_from_host();
    /* the pictures of the coming step: lanes whose chain has ended take the next chain (and forget their reference) */
    auto collect = [&](std::vector<PicRef> &dst, std::vector<int> &lane, std::vector<int> &which, bool commit) {
        int m = 0;
        int nc = next_chain;
        for (int i = 0; i < L; i++) {
            int t = at[(size_t) i], en = end[(size_t) i];
            if (t < 0 || t >= en) {
                if (nc >= k1) {
                    continue;
                }
                t = c.chain_first[(size_t) nc];
                en = c.chain_first[(size_t) nc + 1];
                nc++;
                if (commit) {
                    eng->reset_lane(i);
                }
            }
            if (commit) {
                at[(size_t) i] = t;
                end[(size_t) i] = en;
            }
            lane[(size_t) m] = i;
            which[(size_t) m] = t;
            dst[(size_t) m] = ps.at(t);
            m++;
        }
        if (commit) {
            next_chain = nc;
        }
        return m;
    };
    int m = collect(src, ids, pic, true);
    if (stream_in && m) {
        eng->prefetch(m, ids.data(), src.data());
    }
    cudaEvent_t ready = ps.upload(pic.data(), m);
    const int mapped = 1; /* cudaMallocHost memory */
    while (m > 0) {
        for (int q = 0; q < m; q++) {
            plan[(size_t) q] = c.plan[(size_t) pic[(size_t) q]];
            sinks[(size_t) q].at = e->h_stage + e->stage_slot * (size_t) ids[(size_t) q];
            sinks[(size_t) q].room = e->stage_slot;
            sinks[(size_t) q].overflow = 0;
            sinks[(size_t) q].mapped = mapped;
        }
        /* which pictures come next (needed now for the prefetch) */
        for (int q = 0; q < m; q++) {
            at[(size_t) ids[(size_t) q]]++;
        }
        const int m_next = collect(nxt, nids, npic, false);
        if (stream_in && m_next) {
            eng->prefetch(m_next, nids.data(), nxt.data());
        }
        eng->wait_event(ready);
        ready = ps.upload(npic.data(), m_next);
        eng->step(m, ids.data(), src.data(), reinterpret_cast<DSV_BUF(*)[2]>(bufs.data()), nb.data(), sinks.data(), plan.data());
        for (int q = 0; q < m; q++) {
            const int t = pic[(size_t) q];
            if (nb[(size_t) q] != 1 || sinks[(size_t) q].overflow || !bufs[(size_t) 2 * q].data) {
                c.err = -1;
                continue;
            }
            const DSV_BUF &b = bufs[(size_t) 2 * q];
            c.pkt[(size_t) t].assign(b.data, b.data + b.len);
            if (!c.info.empty()) {
                c.info[(size_t) t] = eng->pic_info[(size_t) q];
            }
            if (!c.ssim.empty()) {
                c.ssim[(size_t) t] = eng->pic_ssim[(size_t) q];
            }
        }
        /* now commit the lane -> chain assignment the prefetch was made for (a lane that takes a new chain forgets
         * its reference only after the last picture of its old chain has been coded) */
        m = collect(src, ids, pic, true);
    }
}

/* gather: metadata + picture packets in order, links patched, EOS */
int long_gather(LongCtx &c, uint8_t *stream, long cap, long *len)
{
    DSV_ENCODER enc;
    apply_cfg(&enc, c.cfg);
    long at = 0;
    unsigned prev_link = 0;
    int rc = c.err;
    auto put = [&](const uint8_t *p, size_t n) {
        if (at + (long) n > cap) {
            rc = -1;
            return (uint8_t *) nullptr;
        }
        uint8_t *dst = stream + at;
        memcpy(dst, p, n);
        at += (long) n;
        return dst;
    };
    for (int t = 0; t < c.nframes && rc == 0; t++) {
        if (c.gop_start[(size_t) t]) {
            DSV_BUF meta;
            make_metadata_packet(&enc, &meta);
            put(meta.data, meta.len);
            dsv_buf_free(&meta);
        }
        const std::vector<uint8_t> &pk = c.pkt[(size_t) t];
        uint8_t *dst = rc == 0 ? put(pk.data(), pk.size()) : nullptr;
        if (dst) { /* set_link_offsets, dsv_encoder.c:170-192 */
            wr_be32(dst + DSV_PACKET_PREV_OFFSET, prev_link);
            wr_be32(dst + DSV_PACKET_NEXT_OFFSET, (unsigned) pk.size());
            prev_link = (unsigned) pk.size();
        }
    }
    if (rc == 0) {
        DSV_BUF eos[1];
        enc.prev_link = (int) prev_link;
        dsv_enc_end_of_stream(&enc, eos);
        put(eos[0].data, eos[0].len);
        dsv_buf_free(&eos[0]);
    }
    *len = rc == 0 ? at : -1;
    return rc;
}

/* a report of a long encode (ctx_init sized it when the report was on) as the records of one sequence */
template <typename R> void take_records(std::vector<R> &recs, int rc, bool *valid, std::vector<std::vector<R>> *out)
{
    *valid = rc == 0 && !recs.empty();
    out->assign(1, std::vector<R>());
    (*out)[0].swap(recs);
}

void fill_info(const LongCtx &c, int *info)
{
    if (info) {
        info[0] = (int) c.chain_first.size() - 1;
        info[1] = c.forced;
        int longest = 0;
        for (size_t k = 0; k + 1 < c.chain_first.size(); k++) {
            const int n = c.chain_first[k + 1] - c.chain_first[k];
            longest = n > longest ? n : longest;
        }
        info[2] = longest;
        info[3] = 0;
    }
}

/* split [0, n) units of the given sizes into `parts` contiguous runs of about equal total size */
std::vector<int> balanced_cuts(const std::vector<int> &sizes, int parts)
{
    long long total = 0;
    for (int s : sizes) {
        total += s;
    }
    std::vector<int> cut((size_t) parts + 1, (int) sizes.size());
    cut[0] = 0;
    long long acc = 0;
    int p = 1;
    for (size_t i = 0; i < sizes.size() && p < parts; i++) {
        acc += sizes[i];
        while (p < parts && acc * parts >= total * p) {
            cut[(size_t) p++] = (int) i + 1;
        }
    }
    return cut;
}

} // namespace

extern "C" int dsvb_encode_long(DSVB_ENC *e, int nframes, const uint8_t *yuv, int on_device, uint8_t *stream, long cap, long *len,
                                int *info)
{
    DSV_API_BEGIN
    if (e->live_open) {
        return -2; /* the chains run on lanes that open live streams hold */
    }
    use_device(e->device);
    e->info_valid = e->ssim_valid = false;
    e->info.clear();
    e->ssim.clear();
    if (nframes <= 0) {
        return -2;
    }
    if (e->cfg[CFG_RC_MODE] != DSV_RATE_CONTROL_CRF) { /* ABR serialises on packet sizes: one lane, like dsv_enc */
        const uint8_t *y[1] = {yuv};
        uint8_t *s[1] = {stream};
        long caps[1] = {cap};
        if (info) {
            info[0] = info[1] = info[2] = 0;
            info[3] = 1;
        }
        return dsvb_encode(e, 1, nframes, y, on_device, s, caps, len);
    }
    LongCtx c;
    ctx_init(c, e, nframes, yuv, on_device);
    PicSource ps;
    ps.open(e, &c);
    long_analyse(e, c, ps, 0, nframes);
    long_decide(c);
    long_code(e, c, ps, 0, (int) c.chain_first.size() - 1);
    fill_info(c, info);
    const int rc = long_gather(c, stream, cap, len);
    take_records(c.info, rc, &e->info_valid, &e->info);
    take_records(c.ssim, rc, &e->ssim_valid, &e->ssim);
    return rc;
    DSV_API_END(-100)
}

extern "C" int dsvb_decode_long(DSVB_DEC *d, const uint8_t *stream, const uint8_t *stream_dev, long len, uint8_t *out, long out_cap,
                                int out_on_device, int *frames)
{
    DSV_API_BEGIN
    if (d->live_open) {
        return -2; /* the chains run on lanes that open live streams hold */
    }
    use_device(d->device);
    /* chains: a new segment starts at every picture without a reference; the metadata packets right in front of it
     * go with it.  Segment 0 holds the stream's first metadata packet and is walked first (lane 0), so the engine
     * exists before a chain that starts with a bare forced I picture is touched. */
    std::vector<DecSegment> segs;
    long at = 0, seg_start = 0, pending_meta = -1;
    bool have_pic = false, seen_meta = false;
    int seg_known = 0, rc = 0;
    auto close = [&](long end) {
        if (end > seg_start) {
            segs.push_back(DecSegment{stream + seg_start, stream_dev ? stream_dev + seg_start : nullptr, end - seg_start, seg_known, out,
                                      out_cap, 0});
        }
    };
    while (at + DSV_PACKET_HDR_SIZE <= len) {
        const uint8_t *hdr = stream + at;
        if (hdr[0] != DSV_FOURCC_0 || hdr[1] != DSV_FOURCC_1 || hdr[2] != DSV_FOURCC_2 || hdr[3] != DSV_FOURCC_3) {
            rc = -4;
            break;
        }
        long size = (long) rd_be32(hdr + DSV_PACKET_NEXT_OFFSET);
        if (size == 0) {
            size = DSV_PACKET_HDR_SIZE;
        }
        if (size < DSV_PACKET_HDR_SIZE || at + size > len) {
            rc = -3;
            break;
        }
        const int type = hdr[DSV_PACKET_TYPE_OFFSET];
        if (type == DSV_PT_META) {
            if (pending_meta < 0) {
                pending_meta = at;
            }
        } else if (type == DSV_PT_EOS) {
            at += size;
            break;
        } else if (DSV_PT_IS_PIC(type)) {
            if (!DSV_PT_HAS_REF(type) && have_pic) {
                const long cut = pending_meta >= 0 ? pending_meta : at;
                close(cut);
                seg_start = cut;
                seg_known = seen_meta ? 1 : 0; /* pictures before any metadata are skipped (dsv_decoder.c:327-331) */
            }
            if (pending_meta >= 0) {
                seen_meta = true;
            }
            have_pic = true;
            pending_meta = -1;
        }
        at += size;
    }
    close(at);
    *frames = 0;
    if (segs.empty()) {
        return rc;
    }
    const int r2 = decode_segments(d, (int) segs.size(), segs.data(), out_on_device);
    for (const DecSegment &s : segs) {
        *frames += s.frames;
    }
    return rc ? rc : r2;
    DSV_API_END(-100)
}

/* ---- several GPUs of one box ---------------------------------------------------------------------- */

struct DSVB_MULTI {
    int ndev = 0, lanes = 0;
    int cfg[CFG_COUNT];
    bool has_cfg = false;
    std::vector<int> devices;
    std::vector<DSVB_ENC *> enc;
    std::vector<DSVB_DEC *> dec;
    bool picture_info = false, picture_ssim = false;
    bool info_valid = false; /* picture report of the last encode call, as DSVB_ENC */
    std::vector<std::vector<DSVB_PICINFO>> info;
    bool ssim_valid = false; /* SSIM report of the last encode call, as DSVB_ENC */
    std::vector<std::vector<DSVB_PICSSIM>> ssim;
};

extern "C" DSVB_MULTI *dsvb_multi_create(const int *cfg, int lanes, int ndev, const int *devices)
{
    DSV_API_BEGIN
    if (ndev < 1 || ndev > 64 || lanes < 1) {
        return nullptr;
    }
    DSVB_MULTI *m = new DSVB_MULTI();
    m->ndev = ndev;
    m->lanes = lanes;
    m->has_cfg = cfg != nullptr;
    if (cfg) {
        memcpy(m->cfg, cfg, sizeof(m->cfg));
    }
    for (int i = 0; i < ndev; i++) {
        m->devices.push_back(devices ? devices[i] : i);
    }
    m->enc.assign((size_t) ndev, nullptr);
    m->dec.assign((size_t) ndev, nullptr);
    return m;
    DSV_API_END(nullptr)
}

extern "C" void dsvb_multi_destroy(DSVB_MULTI *m)
{
    if (!m) {
        return;
    }
    for (DSVB_ENC *e : m->enc) {
        dsvb_enc_destroy(e);
    }
    for (DSVB_DEC *d : m->dec) {
        dsvb_dec_destroy(d);
    }
    delete m;
}

namespace {

/* run f(i) for every device on its own host thread (the engines are per device and per thread) */
template <class F> void per_device(DSVB_MULTI *m, int n, F f)
{
    if (n <= 1) {
        if (n == 1) {
            f(0);
        }
        return;
    }
    std::vector<std::thread> th;
    for (int i = 0; i < n; i++) {
        th.emplace_back([&f, i] { f(i); });
    }
    for (auto &t : th) {
        t.join();
    }
}

bool multi_encoders(DSVB_MULTI *m)
{
    if (!m->has_cfg) {
        return false;
    }
    std::vector<int> ok((size_t) m->ndev, 1);
    per_device(m, m->ndev, [&](int i) {
        if (!m->enc[(size_t) i]) {
            m->enc[(size_t) i] = dsvb_enc_create(m->cfg, m->lanes, m->devices[(size_t) i]);
        }
        ok[(size_t) i] = m->enc[(size_t) i] != nullptr;
        if (ok[(size_t) i]) {
            m->enc[(size_t) i]->eng->picture_info = m->picture_info;
            m->enc[(size_t) i]->eng->picture_ssim = m->picture_ssim;
        }
    });
    for (int v : ok) {
        if (!v) {
            return false;
        }
    }
    return true;
}

void multi_decoders(DSVB_MULTI *m)
{
    for (int i = 0; i < m->ndev; i++) {
        if (!m->dec[(size_t) i]) {
            m->dec[(size_t) i] = dsvb_dec_create(m->lanes, m->devices[(size_t) i]);
        }
    }
}

} // namespace

extern "C" void dsvb_multi_set_picture_info(DSVB_MULTI *m, int on)
{
    m->picture_info = on != 0;
    for (DSVB_ENC *e : m->enc) {
        if (e) {
            e->eng->picture_info = m->picture_info;
        }
    }
}

extern "C" int dsvb_multi_picture_info(DSVB_MULTI *m, int seq, DSVB_PICINFO *out, int cap)
{
    return copy_records(m->info_valid, m->info, seq, out, cap);
}

extern "C" void dsvb_multi_set_picture_ssim(DSVB_MULTI *m, int on)
{
    m->picture_ssim = on != 0;
    for (DSVB_ENC *e : m->enc) {
        if (e) {
            e->eng->picture_ssim = m->picture_ssim;
        }
    }
}

extern "C" int dsvb_multi_picture_ssim(DSVB_MULTI *m, int seq, DSVB_PICSSIM *out, int cap)
{
    return copy_records(m->ssim_valid, m->ssim, seq, out, cap);
}

/* whole sequences dealt to the GPUs in contiguous runs */
extern "C" int dsvb_multi_encode(DSVB_MULTI *m, int nseq, int nframes, const uint8_t *const *yuv, uint8_t *const *streams,
                                 const long *caps, long *lens)
{
    DSV_API_BEGIN
    m->info_valid = m->ssim_valid = false;
    m->info.clear();
    m->ssim.clear();
    if (!multi_encoders(m)) {
        return -100;
    }
    const int nd = m->ndev < nseq ? m->ndev : nseq;
    std::vector<int> rc((size_t) m->ndev, 0);
    per_device(m, nd, [&](int i) {
        const int s0 = (int) ((long long) nseq * i / nd), s1 = (int) ((long long) nseq * (i + 1) / nd);
        rc[(size_t) i] = dsvb_encode(m->enc[(size_t) i], s1 - s0, nframes, yuv + s0, 0, streams + s0, caps + s0, lens + s0);
    });
    for (int v : rc) {
        if (v) {
            return v;
        }
    }
    /* device i coded sequences [s0, s1) as its sequences 0 .. s1 - s0 - 1 */
    m->info.resize(m->picture_info ? (size_t) nseq : 0);
    m->ssim.resize(m->picture_ssim ? (size_t) nseq : 0);
    for (int i = 0; i < nd; i++) {
        const int s0 = (int) ((long long) nseq * i / nd), s1 = (int) ((long long) nseq * (i + 1) / nd);
        for (int s = s0; s < s1; s++) {
            if (m->picture_info) {
                m->info[(size_t) s].swap(m->enc[(size_t) i]->info[(size_t) (s - s0)]);
            }
            if (m->picture_ssim) {
                m->ssim[(size_t) s].swap(m->enc[(size_t) i]->ssim[(size_t) (s - s0)]);
            }
        }
    }
    m->info_valid = m->picture_info;
    m->ssim_valid = m->picture_ssim;
    return 0;
    DSV_API_END(-100)
}

extern "C" int dsvb_multi_decode(DSVB_MULTI *m, int nseq, const uint8_t *const *streams, const long *lens, uint8_t *const *out,
                                 const long *out_caps, int *frames)
{
    DSV_API_BEGIN
    multi_decoders(m);
    const int nd = m->ndev < nseq ? m->ndev : nseq;
    std::vector<int> rc((size_t) m->ndev, 0);
    per_device(m, nd, [&](int i) {
        const int s0 = (int) ((long long) nseq * i / nd), s1 = (int) ((long long) nseq * (i + 1) / nd);
        rc[(size_t) i] = dsvb_decode(m->dec[(size_t) i], s1 - s0, streams + s0, nullptr, lens + s0, out + s0, out_caps + s0, 0, frames + s0);
    });
    for (int v : rc) {
        if (v) {
            return v;
        }
    }
    return 0;
    DSV_API_END(-100)
}

/* one long sequence: phase A over contiguous runs of pictures, phase C over contiguous runs of chains */
extern "C" int dsvb_multi_encode_long(DSVB_MULTI *m, int nframes, const uint8_t *yuv, uint8_t *stream, long cap, long *len, int *info)
{
    DSV_API_BEGIN
    m->info_valid = m->ssim_valid = false;
    m->info.clear();
    m->ssim.clear();
    if (!multi_encoders(m) || nframes <= 0) {
        return -100;
    }
    if (m->cfg[CFG_RC_MODE] != DSV_RATE_CONTROL_CRF || m->ndev == 1) {
        const int rc = dsvb_encode_long(m->enc[0], nframes, yuv, 0, stream, cap, len, info);
        m->info_valid = m->enc[0]->info_valid;
        m->info.swap(m->enc[0]->info);
        m->ssim_valid = m->enc[0]->ssim_valid;
        m->ssim.swap(m->enc[0]->ssim);
        return rc;
    }
    LongCtx c;
    ctx_init(c, m->enc[0], nframes, yuv, 0);
    const int nd = m->ndev < nframes ? m->ndev : nframes;
    std::vector<int> fail((size_t) m->ndev, 0);
    /* phase A: device i analyses pictures [f0, f1) (and uploads [f0 - 1, f1) into its cache) */
    std::vector<PicSource> ps((size_t) nd);
    per_device(m, nd, [&](int i) {
        try {
            DSVB_ENC *e = m->enc[(size_t) i];
            use_device(e->device);
            const int f0 = (int) ((long long) nframes * i / nd), f1 = (int) ((long long) nframes * (i + 1) / nd);
            ps[(size_t) i].open(e, &c);
            long_analyse(e, c, ps[(size_t) i], f0, f1);
        } catch (...) {
            fail[(size_t) i] = 1;
        }
    });
    for (int v : fail) {
        if (v) {
            return -100;
        }
    }
    long_decide(c);
    /* phase C: contiguous runs of chains with about the same number of pictures; most of a run's pictures are
     * already in that device's cache from phase A, the others are read from the host */
    const int nchains = (int) c.chain_first.size() - 1;
    std::vector<int> sizes((size_t) nchains);
    for (int k = 0; k < nchains; k++) {
        sizes[(size_t) k] = c.chain_first[(size_t) k + 1] - c.chain_first[(size_t) k];
    }
    const std::vector<int> cut = balanced_cuts(sizes, nd);
    per_device(m, nd, [&](int i) {
        try {
            DSVB_ENC *e = m->enc[(size_t) i];
            use_device(e->device);
            long_code(e, c, ps[(size_t) i], cut[(size_t) i], cut[(size_t) i + 1]);
        } catch (...) {
            fail[(size_t) i] = 1;
        }
    });
    for (int v : fail) {
        if (v) {
            return -100;
        }
    }
    fill_info(c, info);
    if (info) {
        info[3] = nd;
    }
    const int rc = long_gather(c, stream, cap, len);
    take_records(c.info, rc, &m->info_valid, &m->info);
    take_records(c.ssim, rc, &m->ssim_valid, &m->ssim);
    return rc;
    DSV_API_END(-100)
}

extern "C" int dsvb_multi_decode_long(DSVB_MULTI *m, const uint8_t *stream, long len, uint8_t *out, long out_cap, int *frames)
{
    DSV_API_BEGIN
    multi_decoders(m);
    /* cut the container into one run of chains per GPU at pictures without a reference; every run but the first
     * is given the stream's first metadata packet by decoding it as two segments (metadata, run) */
    struct Pk { long at, size; int type; };
    std::vector<Pk> pk;
    long at = 0;
    while (at + DSV_PACKET_HDR_SIZE <= len) {
        const uint8_t *hdr = stream + at;
        if (hdr[0] != DSV_FOURCC_0 || hdr[1] != DSV_FOURCC_1 || hdr[2] != DSV_FOURCC_2 || hdr[3] != DSV_FOURCC_3) {
            return -4;
        }
        long size = (long) rd_be32(hdr + DSV_PACKET_NEXT_OFFSET);
        if (size == 0) {
            size = DSV_PACKET_HDR_SIZE;
        }
        if (size < DSV_PACKET_HDR_SIZE || at + size > len) {
            return -3;
        }
        pk.push_back(Pk{at, size, hdr[DSV_PACKET_TYPE_OFFSET]});
        at += size;
        if (pk.back().type == DSV_PT_EOS) {
            break;
        }
    }
    /* candidate cut points: metadata packets that directly precede a picture without a reference (GOP starts) */
    std::vector<long> cuts;
    std::vector<int> pics_before; /* pictures in front of each cut */
    int npic = 0;
    for (size_t i = 0; i < pk.size(); i++) {
        if (pk[i].type == DSV_PT_META && i + 1 < pk.size() && DSV_PT_IS_PIC(pk[i + 1].type) && !DSV_PT_HAS_REF(pk[i + 1].type)) {
            cuts.push_back(pk[i].at);
            pics_before.push_back(npic);
        }
        if (DSV_PT_IS_PIC(pk[i].type)) {
            npic++;
        }
    }
    *frames = 0;
    if (cuts.empty() || npic == 0) {
        return dsvb_decode_long(m->dec[0], stream, nullptr, len, out, out_cap, 0, frames);
    }
    const int nd = m->ndev;
    std::vector<long> begin, end;
    {
        size_t ci = 0;
        long b = cuts[0];
        for (int i = 1; i <= nd; i++) {
            const long long want = (long long) npic * i / nd;
            while (ci + 1 < cuts.size() && pics_before[ci + 1] <= want) {
                ci++;
            }
            const long e = (i == nd) ? at : cuts[ci];
            if (e > b) {
                begin.push_back(b);
                end.push_back(e);
                b = e;
            }
        }
    }
    const int nr = (int) begin.size();
    std::vector<int> rc((size_t) nr, 0), got((size_t) nr, 0);
    per_device(m, nr, [&](int i) {
        rc[(size_t) i] = dsvb_decode_long(m->dec[(size_t) i], stream + begin[(size_t) i], nullptr, end[(size_t) i] - begin[(size_t) i], out,
                                          out_cap, 0, &got[(size_t) i]);
    });
    int r = 0;
    for (int i = 0; i < nr; i++) {
        *frames += got[(size_t) i];
        if (rc[(size_t) i] && !r) {
            r = rc[(size_t) i];
        }
    }
    return r;
    DSV_API_END(-100)
}
