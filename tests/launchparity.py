"""Checks of the transform and entropy-coding kernels as the engines launch them (include/dsv1_b200_kernels.h, batch entry
points): tile flags, list scratch, fused prediction add, multi-picture job mapping, carried decoder state.  Shared by
test_emu_launch_parity.py (CPU emulation) and test_gpu_launch_parity.py (B200).  The checkers are the plain-C port
(fwd_sbt, inv_sbt, encode_plane, decode_plane) and numpy, nothing else."""
import ctypes as C

import numpy as np

import dsvlibs as L
from dsvlibs import ptr, i32p

GUARD = 4096  # bytes past the largest cap that the packet buffer exposes (DSVK_PKT_GUARD)


class PIC(C.Structure):
    _fields_ = [("isP", C.c_int), ("quant", C.c_int), ("stable", C.c_void_p), ("start_byte", C.c_uint), ("cap", C.c_uint)]


def quant_of_qp(qp):
    """CRF quality -> frame quantiser (dsv_encoder.c:165): qp 85 -> 313, qp 100 -> 5."""
    q = L.MAX_QUALITY * qp // 100
    return L.MAX_QUALITY - ((L.MAX_QUALITY - 5) * q // L.MAX_QUALITY)


class Geom:
    def __init__(self, w, h, fmt):
        self.w, self.h, self.fmt = w, h, fmt
        self.subsamp = L.SUBSAMP[fmt]
        self.planes = L.plane_dims(w, h, self.subsamp)
        self.coefs = L.coef_dims(w, h, self.subsamp)
        self.frame_bytes = L.frame_bytes(w, h, self.subsamp)
        self.coef_total = sum(cw * ch for cw, ch in self.coefs)
        self.tiles = [(-(-cw // 128), -(-ch // 64)) for cw, ch in self.coefs]
        self.total_tiles = sum(tx * ty for tx, ty in self.tiles)
        self.bw, self.bh, self.nbh, self.nbv = L.block_dims(w, h)

    def split_frame(self, f):
        out, o = [], 0
        for pw, ph in self.planes:
            out.append(f[o:o + pw * ph].reshape(ph, pw))
            o += pw * ph
        return out

    def split_coef(self, c):
        out, o = [], 0
        for cw, ch in self.coefs:
            out.append(c[o:o + cw * ch].reshape(ch, cw))
            o += cw * ch
        return out

    def split_flags(self, t):
        out, o = [], 0
        for tx, ty in self.tiles:
            out.append(t[o:o + tx * ty].reshape(ty, tx))
            o += tx * ty
        return out


def _pics(pics):
    arr = (PIC * len(pics))()
    keep = []
    for a, p in zip(arr, pics):
        a.isP, a.quant = int(p["isP"]), int(p["quant"])
        st = np.ascontiguousarray(p.get("stable", np.zeros(1, np.uint8)), dtype=np.uint8)
        keep.append(st)
        a.stable = st.ctypes.data
        a.start_byte, a.cap = int(p.get("start_byte", 0)), int(p.get("cap", 0))
    return arr, keep


class Enc:
    def __init__(self, lib, g, max_pics):
        self.wrap, self.lib, self.g = lib, lib.lib, g
        self.lib.dsvk_enc_create.restype = C.c_void_p
        self.lib.dsvk_enc_pkt_bytes.restype = C.c_long
        self.h = C.c_void_p(self.lib.dsvk_enc_create(g.w, g.h, g.subsamp, g.bw, g.bh, max_pics))
        assert self.h.value
        self.pkt_bytes = self.lib.dsvk_enc_pkt_bytes(self.h)
        self.dv_pitch = 2 * (g.w + g.h) + 16

    def run(self, pics, frames, preds=None):
        g, n = self.g, len(pics)
        arr, keep = _pics(pics)
        inp = np.ascontiguousarray(np.concatenate(frames), dtype=np.uint8)
        pr = np.ascontiguousarray(np.concatenate(preds), dtype=np.uint8) if preds is not None else None
        pkt = np.full((n, self.pkt_bytes + GUARD), 0xA5, dtype=np.uint8)
        info = np.zeros((n, 8), dtype=np.uint32)
        coef = np.zeros((n, g.coef_total), dtype=np.int32)
        dv = np.zeros((n, 3, self.dv_pitch), dtype=np.int32)
        tfl = np.zeros((n, g.total_tiles), dtype=np.uint8)
        rec = np.zeros((n, g.frame_bytes), dtype=np.uint8)
        rc = self.lib.dsvk_enc_run(self.h, n, arr, ptr(inp), ptr(pr) if pr is not None else None, ptr(pkt),
                                   info.ctypes.data_as(C.POINTER(C.c_uint)), ptr(coef, i32p), ptr(dv, i32p), ptr(tfl), ptr(rec))
        assert rc == 0, rc
        return dict(pkt=pkt, info=info, coef=coef, dv=dv, tflags=tfl, recon=rec)

    def close(self):
        if self.h:
            self.lib.dsvk_enc_destroy(self.h)
            self.h = None


def inv_batch(lib, geoms, pics, coefs, tflags=None, preds=None):
    n = len(pics)
    geo = (C.c_int * (3 * n))(*[v for g in geoms for v in (g.w, g.h, g.subsamp)])
    arr, keep = _pics(pics)
    co = np.ascontiguousarray(np.concatenate([c.ravel() for c in coefs]), dtype=np.int32)
    tf = np.ascontiguousarray(np.concatenate([t.ravel() for t in tflags]), dtype=np.uint8) if tflags is not None else None
    pr = np.ascontiguousarray(np.concatenate(preds), dtype=np.uint8) if preds is not None else None
    out = np.zeros(sum(g.frame_bytes for g in geoms), dtype=np.uint8)
    rc = lib.lib.dsvk_inv_batch(n, geo, arr, ptr(co, i32p), ptr(tf) if tf is not None else None,
                                ptr(pr) if pr is not None else None, ptr(out))
    assert rc == 0, rc
    res, o = [], 0
    for g in geoms:
        res.append(out[o:o + g.frame_bytes])
        o += g.frame_bytes
    return res


class Dec:
    def __init__(self, lib, g):
        self.lib, self.g = lib.lib, g
        self.lib.dsvk_dec_create.restype = C.c_void_p
        self.h = C.c_void_p(self.lib.dsvk_dec_create(g.w, g.h, g.subsamp, g.bw, g.bh))
        assert self.h.value

    def run(self, pic, planes):
        g = self.g
        arr, keep = _pics([pic])
        buf = np.ascontiguousarray(np.frombuffer(planes, dtype=np.uint8))
        coef = np.zeros(g.coef_total, dtype=np.int32)
        tfl = np.zeros(g.total_tiles, dtype=np.uint8)
        n = self.lib.dsvk_dec_run(self.h, arr, ptr(buf), len(buf), ptr(coef, i32p), ptr(tfl))
        assert n >= 0, n
        return n, coef, tfl

    def close(self):
        if self.h:
            self.lib.dsvk_dec_destroy(self.h)
            self.h = None


# ---- numpy references ------------------------------------------------------------------------------------------------
def exact_flags(co):
    """Tile flags a coefficient plane calls for: bit 0 of tile (tx, ty) = a non-zero in the 64x32 block (tx, ty) of
    LH1/HL1/HH1, bit 1 = in the 32x16 block (tx, ty) of LH2/HL2/HH2."""
    ch, cw = co.shape
    tx, ty = -(-cw // 128), -(-ch // 64)
    wo1, ho1 = -(-cw // 2), -(-ch // 2)
    wo2, ho2 = -(-wo1 // 2), -(-ho1 // 2)
    nz = co != 0
    out = np.zeros((ty, tx), dtype=np.uint8)
    for bit, (bw, bh, bands) in ((1, (64, 32, [nz[:ho1, wo1:], nz[ho1:, :wo1], nz[ho1:, wo1:]])),
                                 (2, (32, 16, [nz[:ho2, wo2:wo1], nz[ho2:ho1, :wo2], nz[ho2:ho1, wo2:wo1]]))):
        for b in bands:
            pad = np.zeros((ty * bh, tx * bw), dtype=bool)
            hh, ww = min(b.shape[0], ty * bh), min(b.shape[1], tx * bw)
            pad[:hh, :ww] = b[:hh, :ww]
            any_ = pad.reshape(ty, bh, tx, bw).any(axis=(1, 3))
            out[any_] |= bit
    return out


def flag_base(cw, ch):
    """hz_flag_base: levels whose band is scanned twice at an odd edge keep their decoder flag set."""
    wo = [cw, -(-cw // 2), -(-cw // 4), -(-cw // 8)]
    ho = [ch, -(-ch // 2), -(-ch // 4), -(-ch // 8)]
    b = 0
    for lvl, bit in ((1, 1), (2, 2)):
        if (wo[lvl] & 1) or (ho[lvl] & 1):
            b |= bit
    return b


def recon_ref(port, co, q, isP, c, pw, ph, pred=None):
    r = port.inv_sbt(co, q, isP, c, pw, ph)
    if pred is None:
        return r
    return np.clip(r.astype(np.int32) + pred.astype(np.int32) - 128, 0, 255).astype(np.uint8)


def port_encode(port, g, frame, pic):
    """The port's forward transform + quantiser + coder of one picture: (plane bytes, dequantised coefs) per plane."""
    res = []
    for c, ((pw, ph), (cw, ch), pix) in enumerate(zip(g.planes, g.coefs, g.split_frame(frame))):
        pad = np.zeros((ph, cw), dtype=np.uint8)
        pad[:, :pw] = pix
        raw = port.fwd_sbt(pad, pw, ph, cw, ch, pic["isP"])
        res.append(port.encode_plane(raw, pic["quant"], pic["isP"], c, pic["stable"], g.nbh, g.nbv))
    return res


def frame_content(g, seed, t, rng):
    """Picture t of the synthetic sequence (oracle/synth.c); below 32 samples, where that generator has no room for its
    objects, a smooth gradient with noise."""
    if g.w >= 32 and g.h >= 32:
        return L.synth_sequence(g.w, g.h, g.fmt, 1, seed, start=t)
    out = []
    for pw, ph in g.planes:
        yy, xx = np.mgrid[0:ph, 0:pw]
        out.append((xx * 7 + yy * 5 + t * 3 + rng.integers(0, 40, size=(ph, pw))).clip(0, 255).astype(np.uint8).ravel())
    return np.concatenate(out)


def content(g, n, seed, qps=(85,), shift=(3, 2)):
    """n pictures of synthetic content; odd pictures are P: residual against the previous picture shifted by `shift`."""
    rng = np.random.default_rng(seed)
    frames = [frame_content(g, seed, i, rng) for i in range(n + 1)]
    pics, ins, preds = [], [], []
    for k in range(n):
        isP = k % 2
        cur = frames[k + 1]
        pred = np.concatenate([np.roll(p, shift, axis=(0, 1)).ravel() for p in g.split_frame(frames[k])])
        if isP:
            ins.append(np.clip(cur.astype(np.int32) - pred + 128, 0, 255).astype(np.uint8))
        else:
            ins.append(cur)
        preds.append(pred)
        pics.append(dict(isP=isP, quant=quant_of_qp(qps[k % len(qps)]),
                         stable=rng.integers(0, 4, size=g.nbh * g.nbv, dtype=np.uint8)))
    return pics, ins, preds


def check_encode(port, enc, pics, ins, preds, out, check=None):
    """Encode parity of one dsvk_enc_run result: packet bytes and zeros, coefficients, flags, reconstruction."""
    g = enc.g
    for k, pic in enumerate(pics):
        if check is not None and k not in check:
            continue
        exp = port_encode(port, g, ins[k], pic)
        sb, cap = pic["start_byte"], pic["cap"]
        info = out["info"][k]
        pkt = out["pkt"][k]
        body = np.concatenate([b for b, _ in exp])
        assert info[0] == 0, f"picture {k}: overflow with cap {cap}"
        assert info[1] == sb + len(body), (k, int(info[1]), sb, len(body))
        assert np.array_equal(pkt[sb:info[1]], body), f"picture {k}: packet bytes differ from the port"
        assert not pkt[:sb].any(), f"picture {k}: bytes written before start_byte {sb}"
        assert not pkt[info[1]:].any(), f"picture {k}: bytes written past the packet's end"
        coefs, flags = g.split_coef(out["coef"][k]), g.split_flags(out["tflags"][k])
        rec = g.split_frame(out["recon"][k])
        pr = g.split_frame(preds[k]) if preds is not None and pic["isP"] else [None] * 3
        for c in range(3):
            (pw, ph), (cw, ch) = g.planes[c], g.coefs[c]
            assert np.array_equal(coefs[c], exp[c][1]), f"picture {k} plane {c}: dequantised coefficients"
            check_enc_flags(flags[c], coefs[c], pic["isP"], f"picture {k} plane {c}")
            want = recon_ref(port, exp[c][1], pic["quant"], pic["isP"], c, pw, ph, pr[c])
            assert np.array_equal(rec[c], want), f"picture {k} plane {c}: reconstruction"
            # the double-visit side buffer: the port keeps no such buffer (it codes the first visits, which the packet
            # comparison above checks); here it must equal the single-plane forward + quantiser entry point's
            if cw < 16 or ch < 16 or k >= 2:
                continue  # the single-plane entry point takes no plane below 16x16; an I and a P picture per call suffice
            pad = np.zeros((ph, cw), dtype=np.uint8)
            pad[:, :pw] = g.split_frame(ins[k])[c]
            _, dv1 = L.fwd_sbt_q(enc.wrap, pad, pw, ph, cw, ch, pic["isP"], c, pic["quant"], pic["stable"], g.nbh, g.nbv)
            assert info[5 + c] == len(dv1) and np.array_equal(out["dv"][k, c, :len(dv1)], dv1), f"picture {k} plane {c}: dv"


def check_enc_flags(fl, co, isP, what):
    """Sound: every block with a non-zero is flagged.  Tight away from the last tile column / row (where odd band sizes
    take the generic path, reported as "may be non-zero"): nothing else is flagged, except level 1 of an I picture,
    which the forward kernel always flags (dense anyway), and levels with double-visited positions (flag_base)."""
    ex = exact_flags(co)
    assert np.array_equal(fl & ex, ex), f"{what}: forward tile flags miss a non-zero block (unsound)\n{fl}\n{ex}"
    tight = ex | (0 if isP else 1) | flag_base(co.shape[1], co.shape[0])
    assert np.array_equal(fl[:-1, :-1], tight[:-1, :-1]), \
        f"{what}: PERFORMANCE REGRESSION, not a correctness bug: flags set on empty interior tiles\n{fl}\n{tight}"


def check_dec_flags(fl, co, what):
    ch, cw = co.shape
    ex = exact_flags(co) | flag_base(cw, ch)
    assert np.array_equal(fl & ex, ex), f"{what}: decoder tile flags miss a non-zero block or the base bits\n{fl}\n{ex}"


# ---- caller coefficients through scan / prefix / pack (dsvk_hz_enc_batch) -------------------------------------------
def hz_enc_batch(lib, g, pics, coefs, tflags=None):
    """coefs: per picture the three raw coefficient planes; returns (packets, info, dequantised coefs, dv)."""
    n = len(pics)
    arr, keep = _pics(pics)
    pkt_bytes = max(p["cap"] for p in pics)
    co = np.ascontiguousarray(np.concatenate([c.ravel() for planes in coefs for c in planes]), dtype=np.int32)
    tf = np.ascontiguousarray(np.concatenate([t.ravel() for fl in tflags for t in fl]), dtype=np.uint8) if tflags is not None else None
    info = np.zeros((n, 8), dtype=np.uint32)
    dv = np.zeros((n, 3, 2 * (g.w + g.h) + 16), dtype=np.int32)
    lib.lib.dsvk_enc_create.restype = C.c_void_p
    lib.lib.dsvk_enc_pkt_bytes.restype = C.c_long
    h = C.c_void_p(lib.lib.dsvk_enc_create(g.w, g.h, g.subsamp, g.bw, g.bh, 1))
    cap_all = lib.lib.dsvk_enc_pkt_bytes(h)
    lib.lib.dsvk_enc_destroy(h)
    assert pkt_bytes <= cap_all
    pkt = np.full((n, cap_all + GUARD), 0xA5, dtype=np.uint8)
    rc = lib.lib.dsvk_hz_enc_batch(g.w, g.h, g.subsamp, g.bw, g.bh, n, arr, ptr(co, i32p), ptr(tf) if tf is not None else None,
                                   ptr(pkt), info.ctypes.data_as(C.POINTER(C.c_uint)), ptr(dv, i32p))
    assert rc == 0, rc
    return pkt, info, co.reshape(n, g.coef_total), dv


def scan_map(cw, ch):
    """(x, y) of every scan position of a plane (hz_fill_regions): LL, then LH / HL / HH of transform levels 3, 2, 1."""
    xs, ys = [], []
    def add(x0, y0, sw, sh):
        yy, xx = np.mgrid[0:sh, 0:sw]
        xs.append((xx + x0).ravel())
        ys.append((yy + y0).ravel())
    add(0, 0, -(-cw // 8), -(-ch // 8))
    for sh_ in (3, 2, 1):
        sw, sh = -(-cw // (1 << sh_)), -(-ch // (1 << sh_))
        add(sw, 0, sw, sh)
        add(0, sh, sw, sh)
        add(sw, sh, sw, sh)
    return np.concatenate(xs), np.concatenate(ys)


CHUNK = 2048


def marked_groups(co, chunk):
    """groups of 4 scan positions of the chunk that hold a non-zero (dequantised) coefficient, and the non-zeros"""
    ch, cw = co.shape
    xs, ys = scan_map(cw, ch)
    v = co[ys[chunk * CHUNK:(chunk + 1) * CHUNK], xs[chunk * CHUNK:(chunk + 1) * CHUNK]] != 0
    v = np.pad(v, (0, CHUNK - len(v)))
    return int(v.reshape(-1, 4).any(axis=1).sum()), int(v.sum())


# Luma chunks of a 384x192 plane (36 chunks: LL + level 3 + level 2 in chunks 0-8, then LH1 9-17, HL1 18-26, HH1
# 27-35; each level-1 band is 192 x 96, tile rows of 32 band rows): what each test chunk holds, as
# (marked groups, non-zeros per group).  Tile row 2 of level 1 (chunks 15-17, 24-26, 33-35) and the level-2 bands stay
# empty, so their chunks are flagged empty next to chunks that are not.
LIST_EDGE_CHUNKS = {9: (127, 1), 11: (128, 1), 13: (129, 1), 18: (127, 4), 21: (128, 4), 22: (129, 4), 31: (40, 2)}
BOUNDARY_POSITIONS = (20 * CHUNK - 1, 20 * CHUNK)  # the last position of chunk 19 and the first of chunk 20


def list_edge_planes(g, rng):
    """raw coefficient planes of a 384x192 4:2:0 picture: the luma chunks above, all-zero chroma planes"""
    cw, ch = g.coefs[0]
    assert (cw, ch) == (384, 192)
    xs, ys = scan_map(cw, ch)
    y = np.zeros((ch, cw), dtype=np.int32)
    def put(pos):
        y[ys[pos], xs[pos]] = int(rng.choice([-1, 1])) * int(rng.integers(1500, 4000))
    for chunk, (groups, per) in LIST_EDGE_CHUNKS.items():
        for gi in rng.choice(CHUNK // 4, size=groups, replace=False):
            for j in (rng.choice(4, size=per, replace=False) if per < 4 else range(4)):
                put(chunk * CHUNK + 4 * int(gi) + int(j))
    for pos in BOUNDARY_POSITIONS:
        put(pos)
    return [y] + [np.zeros((c[1], c[0]), dtype=np.int32) for c in g.coefs[1:]]
