"""Live streams of the batch objects (dsvb_enc_open / _push / _close, dsvb_dec_open / _push / _close,
include/dsv1_b200_batch.h) from Python, and the drivers the tests share.

LiveEncoder / LiveDecoder extend dsvlibs.BatchEncoder / BatchDecoder (same handle, so the batch calls and the reports
work on them too).  live_encode / live_decode run several streams through one object with staggered opens and a
random subset of the open streams in every push.  Used by test_emu_live.py (CPU emulation), test_gpu_live.py (B200)
and tools/live_rate.py."""
import ctypes as C

import numpy as np

import dsvlibs as L

DEC_OK, DEC_ERROR, DEC_EOS, DEC_GOT_META = 0, 1, 2, 3   # DSV_DEC_* (dsv1_b200.h)
HDR = 14                                               # DSV_PACKET_HDR_SIZE
PT_META, PT_EOS = 0x00, 0x10


def _arr(ty, vals):
    return (ty * len(vals))(*vals)


class LiveEncoder(L.BatchEncoder):
    def __init__(self, lib, cfg, lanes, device=0):
        super().__init__(lib, cfg, lanes, device)
        self.lib.dsvb_enc_push_bound.restype = C.c_long
        self.bound = self.lib.dsvb_enc_push_bound(self.h)

    def open(self):
        return self.lib.dsvb_enc_open(self.h)

    def push_ptrs(self, ids, pic_ptrs, on_device, out_ptrs, caps):
        """raw call: returns (rc, lens)"""
        n = len(ids)
        lens = (C.c_long * n)()
        rc = self.lib.dsvb_enc_push(self.h, n, _arr(C.c_int, ids), _arr(C.c_void_p, pic_ptrs), int(on_device),
                                    _arr(C.c_void_p, out_ptrs), _arr(C.c_long, caps), lens)
        return rc, list(lens)

    def push(self, ids, pics, on_device=False, caps=None):
        """pics: host numpy pictures, or device addresses with on_device.  Returns (rc, [bytes, or None where lens = -1])"""
        caps = caps or [self.bound] * len(ids)
        outs = [np.zeros(max(c, 1), dtype=np.uint8) for c in caps]
        ptrs = [p if isinstance(p, int) else p.ctypes.data for p in pics]
        rc, lens = self.push_ptrs(ids, ptrs, on_device, [o.ctypes.data for o in outs], caps)
        return rc, [o[:n].tobytes() if n >= 0 else None for o, n in zip(outs, lens)]

    def end(self, sid, cap=64):
        """dsvb_enc_close: (rc, EOS bytes or None)"""
        out = np.zeros(max(cap, 1), dtype=np.uint8)
        ln = C.c_long(0)
        rc = self.lib.dsvb_enc_close(self.h, int(sid), C.c_void_p(out.ctypes.data) if cap else None, C.c_long(cap), C.byref(ln))
        return rc, out[:ln.value].tobytes() if ln.value >= 0 else None


class LiveDecoder(L.BatchDecoder):
    def open(self):
        return self.lib.dsvb_dec_open(self.h)

    def end(self, sid):
        self.lib.dsvb_dec_close(self.h, int(sid))

    def push_ptrs(self, ids, pkt_ptrs, dev_ptrs, lens, out_ptrs, out_on_device):
        """raw call: returns (rc, codes, fnums)"""
        n = len(ids)
        codes = (C.c_int * n)()
        fnums = (C.c_longlong * n)()
        rc = self.lib.dsvb_dec_push(self.h, n, _arr(C.c_int, ids), _arr(C.c_void_p, pkt_ptrs),
                                    _arr(C.c_void_p, dev_ptrs) if dev_ptrs is not None else None, _arr(C.c_long, lens),
                                    _arr(C.c_void_p, out_ptrs) if out_ptrs is not None else None, int(out_on_device), codes, fnums)
        return rc, list(codes), list(fnums)

    def push(self, ids, pkts, frame_bytes):
        """one packet (bytes) per stream, pictures to fresh host buffers: (rc, codes, fnums, pictures)"""
        bufs = [np.frombuffer(p, dtype=np.uint8) for p in pkts]
        outs = [np.zeros(frame_bytes, dtype=np.uint8) for _ in pkts]
        rc, codes, fnums = self.push_ptrs(ids, [b.ctypes.data for b in bufs], None, [len(b) for b in bufs],
                                          [o.ctypes.data for o in outs], 0)
        return rc, codes, fnums, outs


def split_packets(stream):
    """a .dsv stream cut into its packets (next links; an EOS packet's link is 0)"""
    out, at = [], 0
    while at + HDR <= len(stream):
        size = int.from_bytes(stream[at + 10:at + 14], "big") or HDR
        out.append(stream[at:at + size])
        at += size
    assert at == len(stream), (at, len(stream))
    return out


def frame(seq, t, fb):
    return seq[t * fb:(t + 1) * fb]


def live_encode(enc, seqs, counts, rng, stagger=1, on_device=False, pics=None, on_push=None):
    """Encode len(seqs) streams through `enc`: stream i opens once i * stagger pushes have been made and a lane is free,
    every push takes a random non-empty subset of the open streams, a stream is closed after its counts[i] pictures.
    seqs[i]: host pictures back to back (or, with on_device, pics(i, t) gives a device address).  on_push(take) runs
    after every push with the stream indices in push order.  Returns the streams as bytes and, per stream, the list of
    (push number, position in that push) of its pictures."""
    fb = L.frame_bytes(enc.cfg[0], enc.cfg[1], enc.cfg[2])
    ns = len(counts)
    out = [b"" for _ in range(ns)]
    where = [[] for _ in range(ns)]
    sid, done = [None] * ns, [0] * ns
    nxt, pushes = 0, 0
    while nxt < ns or any(s is not None for s in sid):
        while nxt < ns and pushes >= nxt * stagger:
            s = enc.open()
            if s < 0:
                break
            sid[nxt] = s
            nxt += 1
        live = [i for i in range(ns) if sid[i] is not None]
        take = [i for i in live if rng.random() < 0.7] or [live[int(rng.integers(len(live)))]]
        rng.shuffle(take)
        src = [pics(i, done[i]) if on_device else frame(seqs[i], done[i], fb) for i in take]
        rc, got = enc.push([sid[i] for i in take], src, on_device=on_device)
        assert rc == 0, rc
        if on_push:
            on_push(take)
        for k, i in enumerate(take):
            out[i] += got[k]
            where[i].append((pushes, k))
            done[i] += 1
            if done[i] == counts[i]:
                rc, eos = enc.end(sid[i])
                assert rc == 0 and len(eos) == HDR
                out[i] += eos
                sid[i] = None
        pushes += 1
    return out, where


def live_decode(dec, streams, frame_bytes, counts, rng):
    """Decode the streams packet by packet through `dec`, interleaved at random; every stream opens at the start and
    closes after its last packet.  Returns each stream's pictures back to back in frame-number order."""
    pk = [split_packets(s) for s in streams]
    pos = [0] * len(streams)
    pics = [np.zeros(frame_bytes * n, dtype=np.uint8) for n in counts]
    sid = [dec.open() for _ in streams]
    assert all(s >= 0 for s in sid)
    while any(p < len(q) for p, q in zip(pos, pk)):
        live = [i for i in range(len(streams)) if pos[i] < len(pk[i])]
        take = [i for i in live if rng.random() < 0.6] or [live[int(rng.integers(len(live)))]]
        rng.shuffle(take)
        rc, codes, fnums, outs = dec.push([sid[i] for i in take], [pk[i][pos[i]] for i in take], frame_bytes)
        assert rc == 0, rc
        for k, i in enumerate(take):
            t = pk[i][pos[i]][5]
            want = DEC_GOT_META if t == PT_META else DEC_EOS if t == PT_EOS else DEC_OK
            assert codes[k] == want, (i, pos[i], codes[k])
            if want == DEC_OK:
                f = fnums[k]
                assert 0 <= f < counts[i]
                pics[i][f * frame_bytes:(f + 1) * frame_bytes] = outs[k]
            pos[i] += 1
            if pos[i] == len(pk[i]):
                dec.end(sid[i])
    return pics


# ---- checks shared by the CPU-emulation and B200 tests ---------------------------------------------------------------

def check_mixed_streams(lib, w, h, fmt, lanes, specs, seed, **cfgkw):
    """More streams than lanes, of different seeds, lengths and scene cuts, opened as lanes free up: pushes mix I and
    P pictures and fresh lanes.  Every stream equals dsv_enc's (lib.encode_sequence) for its pictures, and decodes
    packet by packet to what dsv_dec gives.  specs: [(pictures, seed, cut)]."""
    sub = L.SUBSAMP[fmt]
    fb = L.frame_bytes(w, h, sub)
    cfg = L.make_cfg(w, h, fmt, **cfgkw)
    seqs = [L.synth_sequence(w, h, fmt, n, s, c) for n, s, c in specs]
    counts = [n for n, _, _ in specs]
    want = [lib.encode_sequence(cfg, q, n)[0] for q, n in zip(seqs, counts)]
    enc = LiveEncoder(lib, cfg, lanes)
    try:
        got, _ = live_encode(enc, seqs, counts, np.random.default_rng(seed), stagger=2)
    finally:
        enc.close()
    for i, (a, b) in enumerate(zip(got, want)):
        assert a == b, i
    dec = LiveDecoder(lib, len(specs))
    try:
        pics = live_decode(dec, want, fb, counts, np.random.default_rng(seed + 1))
    finally:
        dec.close()
    for s, n, p in zip(want, counts, pics):
        nf, d, _, _ = lib.decode_stream(s, w, h, sub, n)
        assert nf == n and np.array_equal(d, p)


def check_reports(lib, w, h, fmt, n, nseq, seed, **cfgkw):
    """The picture info and SSIM records a stream collects push by push equal, in order, those dsvb_encode gives for
    the same sequence."""
    import picinfo as PI
    import picssim as PS
    cfg = L.make_cfg(w, h, fmt, **cfgkw)
    seqs = [L.synth_sequence(w, h, fmt, n, seed + s, 3 if s == 1 else 0) for s in range(nseq)]
    be = L.BatchEncoder(lib, cfg, nseq)
    PI.set_picture_info(be, 1)
    PS.set_picture_ssim(be, 1)
    want = be.encode(seqs, n)
    want_info = [PI.picture_info(be, s) for s in range(nseq)]
    want_ssim = [PS.picture_ssim(be, s) for s in range(nseq)]
    be.close()
    enc = LiveEncoder(lib, cfg, nseq)
    PI.set_picture_info(enc, 1)
    PS.set_picture_ssim(enc, 1)
    info, ssim = [[] for _ in seqs], [[] for _ in seqs]

    def collect(take):
        assert PI.picture_info(enc, len(take)) is None and PS.picture_ssim(enc, -1) is None
        for k, i in enumerate(take):
            a, b = PI.picture_info(enc, k), PS.picture_ssim(enc, k)
            assert len(a) == 1 and len(b) == 1
            info[i].append(a[0])
            ssim[i].append(b[0])
    try:
        got, _ = live_encode(enc, seqs, [n] * nseq, np.random.default_rng(seed), stagger=1, on_push=collect)
    finally:
        enc.close()
    assert got == want
    for s in range(nseq):
        assert np.array(info[s], dtype=PI.PICINFO_DTYPE).tobytes() == want_info[s].tobytes(), s
        assert np.array(ssim[s], dtype=PS.PICSSIM_DTYPE).tobytes() == want_ssim[s].tobytes(), s


def check_encoder_errors(lib, w, h, fmt):
    """open beyond the lanes; closed, duplicate and out-of-range ids refused with nothing consumed; a too-small output
    breaks that stream only; the batch calls refused while a stream is open and fine after the last close."""
    sub = L.SUBSAMP[fmt]
    fb = L.frame_bytes(w, h, sub)
    cfg = L.make_cfg(w, h, fmt, gop=4)
    n = 7
    seq = L.synth_sequence(w, h, fmt, n, 71, 5)
    other = L.synth_sequence(w, h, fmt, 2, 72, 0)
    want = lib.encode_sequence(cfg, seq, n)[0]
    enc = LiveEncoder(lib, cfg, 2)
    try:
        a, b = enc.open(), enc.open()
        assert (a, b) == (0, 1) and enc.open() == -1
        got = b""
        t = 0
        step = enc.push
        assert step([a, a], [frame(seq, 0, fb)] * 2)[0] == -2
        assert step([2], [frame(seq, 0, fb)])[0] == -2 and step([-1], [frame(seq, 0, fb)])[0] == -2
        rc, out = step([a], [frame(seq, t, fb)])
        assert rc == 0
        got += out[0]
        t += 1
        rc, eos = enc.end(b)
        assert rc == 0 and len(eos) == HDR
        # b is closed now: a push naming it is refused whole, a's next picture is not consumed
        assert enc.end(b)[0] == -2
        assert step([a, b], [frame(seq, t, fb), frame(other, 0, fb)])[0] == -2
        # the batch calls refuse to run while a stream is open
        s = np.zeros(1 << 20, dtype=np.uint8)
        assert enc.encode_ptrs([other.ctypes.data], 1, 0, [s.ctypes.data], [len(s)])[0] == -2
        assert enc.encode_long_ptr(other.ctypes.data, 1, 0, s.ctypes.data, len(s))[0] == -2
        # a too-small output: that stream breaks (lens -1, later pushes -2), the other one is complete
        c = enc.open()
        assert c == 1
        rc, out = step([c, a], [frame(other, 0, fb), frame(seq, t, fb)], caps=[20, enc.bound])
        assert rc == -1 and out[0] is None and out[1] is not None
        got += out[1]
        t += 1
        assert step([c], [frame(other, 1, fb)])[0] == -2
        assert enc.end(c, cap=0) == (-1, None)       # closed all the same: the lane is free again
        assert enc.open() == 1
        assert enc.end(1)[0] == 0
        while t < n:
            rc, out = step([a], [frame(seq, t, fb)])
            assert rc == 0
            got += out[0]
            t += 1
        rc, eos = enc.end(a)
        assert rc == 0
        assert got + eos == want
        # every stream closed: the batch call works again and gives the same stream
        rc, lens = enc.encode_ptrs([seq.ctypes.data], n, 0, [s.ctypes.data], [len(s)])
        assert rc == 0 and s[:lens[0]].tobytes() == want
    finally:
        enc.close()


def check_decoder_errors(lib, w, h, fmt, w2, h2):
    """pictures before metadata skipped with fnum -1; a P picture without its reference is an error; a metadata packet
    of another format is refused while another stream holds the format, accepted once none does; the batch calls
    refused while a stream is open; duplicate and closed ids refused."""
    sub = L.SUBSAMP[fmt]
    fb = L.frame_bytes(w, h, sub)
    cfg = L.make_cfg(w, h, fmt, gop=4)
    seq = L.synth_sequence(w, h, fmt, 3, 81, 0)
    stream = lib.encode_sequence(cfg, seq, 3)[0]
    pk = split_packets(stream)                  # META I P P EOS
    assert [p[5] for p in pk][0] == PT_META and len(pk) == 5
    _, ref, _, _ = lib.decode_stream(stream, w, h, sub, 3)
    other = lib.encode_sequence(L.make_cfg(w2, h2, fmt, gop=4), L.synth_sequence(w2, h2, fmt, 1, 82, 0), 1)[0]
    opk = split_packets(other)
    dec = LiveDecoder(lib, 2)
    try:
        a = dec.open()
        rc, codes, fn, _ = dec.push([a], [pk[1]], fb)
        assert rc == 0 and codes == [DEC_OK] and fn == [-1]          # no metadata yet: skipped
        assert dec.push([a], [pk[0]], fb)[1] == [DEC_GOT_META]
        rc, codes, fn, _ = dec.push([a], [pk[2]], fb)
        assert codes == [DEC_ERROR] and fn == [1]                     # P picture, no reference
        assert dec.push([a, a], [pk[1], pk[1]], fb)[0] == -2
        assert dec.push([1], [pk[1]], fb)[0] == -2 and dec.push([7], [pk[1]], fb)[0] == -2
        b = dec.open()
        assert dec.open() == -1
        rc, codes, fn, outs = dec.push([b, a], [opk[0], pk[1]], fb)   # b: another format while a holds one
        assert rc == 0 and codes == [DEC_ERROR, DEC_OK] and fn[1] == 0 and np.array_equal(outs[1], ref[:fb])
        assert dec.push([b], [pk[1]], fb)[1:3] == ([DEC_OK], [-1])    # b stayed without a format
        assert dec.push([b], [b"XXXX" + pk[1][4:]], fb)[1] == [DEC_ERROR]
        s = np.frombuffer(stream, dtype=np.uint8)
        o = np.zeros(fb * 3, dtype=np.uint8)
        assert dec.decode_ptrs([s.ctypes.data], None, [len(s)], [o.ctypes.data], [len(o)], 0)[0] == -2
        rc, codes, fn, outs = dec.push([a], [pk[2]], fb)
        assert codes == [DEC_OK] and fn == [1] and np.array_equal(outs[0], ref[fb:2 * fb])
        assert dec.push([a], [pk[4]], fb)[1] == [DEC_EOS]
        dec.end(a)
        # b is the only stream left and has no format: the other format replaces the engine
        fb2 = L.frame_bytes(w2, h2, sub)
        assert dec.push([b], [opk[0]], fb2)[1] == [DEC_GOT_META]
        rc, codes, fn, outs = dec.push([b], [opk[1]], fb2)
        _, oref, _, _ = lib.decode_stream(other, w2, h2, sub, 1)
        assert codes == [DEC_OK] and fn == [0] and np.array_equal(outs[0], oref)
        dec.end(b)
        dec.end(b)                                                  # closing twice is harmless
        assert dec.push([b], [opk[1]], fb2)[0] == -2
        rc, fr = dec.decode_ptrs([s.ctypes.data], None, [len(s)], [o.ctypes.data], [len(o)], 0)
        assert rc == 0 and fr == [3] and np.array_equal(o, ref)
    finally:
        dec.close()
