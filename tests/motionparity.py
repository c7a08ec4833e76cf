"""Checks of the motion kernels as the engines launch them (include/dsv1_b200_kernels.h, dsvk_me_* and
dsvk_add_pred_batch): ingest with its replicated border, the batched pyramid, luma sum and zeroing, the search over
several lanes with the engine's argument layout and reference ping-pong, the encoder's out-of-place compensation from
the reconstruction, the long encode's code pass and the decoder's in-place compensation.  Shared by
test_emu_motion_parity.py (CPU emulation) and test_gpu_motion_parity.py (B200).  The checkers are the plain-C port
(pyramid, hme, sub_pred, add_pred) and numpy, nothing else."""
import ctypes as C
import math

import numpy as np

import dsvlibs as L
from dsvlibs import ptr

BORDER = 64
GUARD = 4 * 4096  # zeroed bytes in front of and behind every device frame (DSV_GUARD_BYTES)
MV_FIELDS = [k for k in L.MV_DTYPE.names if k != "pad"]


class MEPIC(C.Structure):
    _fields_ = [("src", C.c_void_p), ("src_on_device", C.c_int), ("stage_offset", C.c_uint), ("has_ref", C.c_int),
                ("do_sum", C.c_int), ("recon", C.c_void_p)]


def frame_stride(w):
    return (w + 2 * BORDER + 15) & ~15


def alloc_bytes(w, h, subsamp):
    """DevFrame::bytes of a w x h frame (frame_ops.cu devframe_alloc)"""
    return sum(frame_stride(pw) * (ph + 2 * BORDER) for pw, ph in L.plane_dims(w, h, subsamp)) + 2 * GUARD


def pyr_levels(w, h, nbh, nbv):
    """dsv_encoder.c:602-613"""
    lv = int(math.ceil(math.log2(min(w, h))))
    while (1 << lv) > max(nbh, nbv):
        lv -= 1
    return min(max(lv, 3), 5)


class Geom:
    def __init__(self, w, h, fmt, blk=None, levels=None):
        self.w, self.h, self.fmt = w, h, fmt
        self.subsamp = L.SUBSAMP[fmt]
        self.planes = L.plane_dims(w, h, self.subsamp)
        self.frame_bytes = L.frame_bytes(w, h, self.subsamp)
        if blk is None:
            self.bw, self.bh = L.block_dims(w, h)[:2]
        else:
            self.bw, self.bh = blk
        self.nbh, self.nbv = -(-w // self.bw), -(-h // self.bh)
        self.nblk = self.nbh * self.nbv
        self.blk = (self.bw, self.bh, self.nbh, self.nbv)
        self.levels = levels if levels is not None else pyr_levels(w, h, self.nbh, self.nbv)
        self.level_dims = [(w, h)] + [(-(-w // (1 << (k + 1))), -(-h // (1 << (k + 1)))) for k in range(self.levels)]
        self.level_bytes = [alloc_bytes(lw, lh, self.subsamp) for lw, lh in self.level_dims]

    def __repr__(self):
        return f"{self.w}x{self.h}_{self.fmt}_{self.bw}x{self.bh}_L{self.levels}"

    def split(self, f):
        out, o = [], 0
        for pw, ph in self.planes:
            out.append(f[o:o + pw * ph].reshape(ph, pw))
            o += pw * ph
        return out


def frame_model(planes, dims):
    """The whole device allocation of a bordered frame: zeros, then each plane's (h + 128) x (w + 128) window at its
    stride holding the plane with its edges replicated 64 samples out.  planes[p] None: that plane was never written."""
    out = np.zeros(sum(frame_stride(pw) * (ph + 2 * BORDER) for pw, ph in dims) + 2 * GUARD, dtype=np.uint8)
    o = GUARD
    for pl, (pw, ph) in zip(planes, dims):
        s = frame_stride(pw)
        if pl is not None:
            win = out[o:o + s * (ph + 2 * BORDER)].reshape(ph + 2 * BORDER, s)
            win[:, :pw + 2 * BORDER] = np.pad(pl, BORDER, mode="edge")
        o += s * (ph + 2 * BORDER)
    return out


def first_diff(a, b):
    d = np.flatnonzero(a != b)
    return f"{len(d)} bytes differ, first at {d[0]} (got {a[d[0]]}, want {b[d[0]]})" if len(d) else "equal"


# ---- the port ------------------------------------------------------------------------------------------------------
def port_hme(port, g, src, ref):
    """(intra percentage, level-0 field) of the port's search of src against ref with g's block grid and levels"""
    mv = np.zeros(g.nblk, dtype=L.MV_DTYPE)
    pct = port.fn("hme")(ptr(np.ascontiguousarray(src)), ptr(np.ascontiguousarray(ref)), g.w, g.h, g.subsamp, g.bw, g.bh,
                         g.levels, ptr(mv.view(np.uint8)))
    return pct, mv


def port_pyramid(port, g, src):
    return port.pyramid(src, g.w, g.h, g.subsamp, g.levels)


def random_field(rng, nblk, amp=110, intra=0.3):
    """vectors up to amp half-pels (110 keeps every filter tap inside the reference's own allocation), a share of intra
    blocks with partial submasks: the fields of test_emu_bmc.test_bmc_strips"""
    mv = np.zeros(nblk, dtype=L.MV_DTYPE)
    mv["x"] = rng.integers(-amp, amp + 1, size=nblk).astype(np.int16)
    mv["y"] = rng.integers(-amp, amp + 1, size=nblk).astype(np.int16)
    mv["mode"] = (rng.random(nblk) < intra).astype(np.uint8)
    mv["submask"] = np.where(mv["mode"] == 1, rng.integers(1, 16, size=nblk), 0).astype(np.uint8)
    return mv


def content(g, seed, t, kind="synth"):
    """picture t of lane content: the synthetic sequence (oracle/synth.c, moving objects), or noise for a lane that must
    not look like its neighbours; below 32 samples a moving gradient with noise"""
    rng = np.random.default_rng(seed * 1000 + t)
    if kind == "noise":
        return rng.integers(0, 256, size=g.frame_bytes, dtype=np.uint8)
    if g.w >= 32 and g.h >= 32:
        return L.synth_sequence(g.w, g.h, g.fmt, 1, seed, start=t)
    out = []
    for pw, ph in g.planes:
        yy, xx = np.mgrid[0:ph, 0:pw]
        out.append((xx * 7 + yy * 5 + t * 3 + rng.integers(0, 40, size=(ph, pw))).clip(0, 255).astype(np.uint8).ravel())
    return np.concatenate(out)


def recon_of(src, seed):
    """a stand-in reconstruction: the picture with coding noise"""
    rng = np.random.default_rng(seed)
    return np.clip(src.astype(np.int32) + rng.integers(-6, 7, size=src.shape), 0, 255).astype(np.uint8)


def at_offset(a, off, align=256):
    """a copy of a whose first byte is `off` bytes past an `align`-byte boundary, and its buffer: in the emulator, whose
    device memory is host memory, a "device-resident" source read where it lies"""
    buf = np.zeros(len(a) + 2 * align, dtype=np.uint8)
    base = (-buf.ctypes.data) % align
    v = buf[base + off:base + off + len(a)]
    v[:] = a
    return v, buf


# ---- the entry points ----------------------------------------------------------------------------------------------
class Me:
    def __init__(self, lib, g, max_pics):
        self.lib, self.g = lib.lib, g
        self.lib.dsvk_me_create.restype = C.c_void_p
        self.lib.dsvk_me_frame_bytes.restype = C.c_long
        self.h = C.c_void_p(self.lib.dsvk_me_create(g.w, g.h, g.subsamp, g.bw, g.bh, g.levels, max_pics))
        assert self.h.value
        got = [self.lib.dsvk_me_frame_bytes(self.h, lv) for lv in range(g.levels + 1)]
        assert got == g.level_bytes, (got, g.level_bytes)
        self.pitch = sum(g.level_bytes)

    def run(self, pics, mvs=None, expect_rc=0):
        """pics: dicts with src (numpy array, or an int device address with on_device=1), on_device, stage_offset,
        has_ref, do_sum, recon (numpy or None).  mvs: None (search) or n fields (code pass)."""
        g, n = self.g, len(pics)
        arr = (MEPIC * n)()
        keep = []
        for a, p in zip(arr, pics):
            src = p["src"]
            if isinstance(src, np.ndarray):
                keep.append(src)
                src = src.ctypes.data
            a.src, a.src_on_device, a.stage_offset = src, int(p.get("on_device", 0)), int(p.get("stage_offset", 0))
            a.has_ref, a.do_sum = int(p["has_ref"]), int(p["do_sum"])
            if p.get("recon") is not None:
                r = np.ascontiguousarray(p["recon"], dtype=np.uint8)
                keep.append(r)
                a.recon = r.ctypes.data
        mv_in = None
        if mvs is not None:
            mv_in = np.ascontiguousarray(np.concatenate(mvs))
        frames = np.full((n, self.pitch), 0x5A, dtype=np.uint8)
        misc = np.full((n, 2), -1, dtype=np.int64)
        mv = np.zeros(n * g.nblk, dtype=L.MV_DTYPE)
        pred = np.zeros((n, g.frame_bytes), dtype=np.uint8)
        resid = np.zeros((n, g.frame_bytes), dtype=np.uint8)
        rc = self.lib.dsvk_me_run(self.h, n, arr, ptr(mv_in.view(np.uint8)) if mv_in is not None else None, ptr(frames),
                                  misc.ctypes.data_as(C.POINTER(C.c_int64)), ptr(mv.view(np.uint8)), ptr(pred), ptr(resid))
        assert rc == expect_rc, rc
        if rc:
            return None
        lv_frames = []
        for k in range(n):
            o, fs = 0, []
            for b in g.level_bytes:
                fs.append(frames[k, o:o + b])
                o += b
            lv_frames.append(fs)
        return dict(frames=lv_frames, misc=misc, mv=mv.reshape(n, g.nblk), pred=pred, resid=resid)

    def close(self):
        if self.h:
            self.lib.dsvk_me_destroy(self.h)
            self.h = None


def add_pred_batch(lib, g, isP, mvs, resid, ref):
    n = len(isP)
    ip = (C.c_int * n)(*[int(v) for v in isP])
    mv = np.ascontiguousarray(np.concatenate(mvs))
    rs = np.ascontiguousarray(np.concatenate(resid), dtype=np.uint8)
    rf = np.ascontiguousarray(np.concatenate(ref), dtype=np.uint8)
    out = np.zeros((n, g.frame_bytes), dtype=np.uint8)
    rc = lib.lib.dsvk_add_pred_batch(g.w, g.h, g.subsamp, g.bw, g.bh, n, ip, ptr(mv.view(np.uint8)), ptr(rs), ptr(rf), ptr(out))
    assert rc == 0, rc
    return out


# ---- the checks ----------------------------------------------------------------------------------------------------
class LaneModel:
    """What a lane holds between calls: its previous source and reconstruction"""

    def __init__(self):
        self.prev_src = None
        self.prev_recon = None


def check_frames(port, g, k, src, got, what):
    """the ingested frame and every pyramid level, whole allocations: interior, replicated border, zero stride tail and
    guard bands; pyramid chroma planes are never written"""
    want0 = frame_model(g.split(src), g.planes)
    assert np.array_equal(got[0], want0), f"{what} lane {k}: ingested frame: {first_diff(got[0], want0)}"
    for lv, lvl in enumerate(port_pyramid(port, g, src)):
        lw, lh = g.level_dims[lv + 1]
        dims = L.plane_dims(lw, lh, g.subsamp)
        want = frame_model([lvl, None, None], dims)
        assert np.array_equal(got[lv + 1], want), f"{what} lane {k}: pyramid level {lv + 1} ({lw}x{lh}): {first_diff(got[lv + 1], want)}"


def check_run(port, g, lanes, pics, out, mvs=None, what="", check=None):
    """compare one dsvk_me_run result with the port; lanes (LaneModel per lane) are advanced"""
    code = mvs is not None
    zeroed = not code and any(p["has_ref"] or p["do_sum"] for p in pics)
    for k, p in enumerate(pics):
        src, lm = p["host_src"], lanes[k]
        if code:  # no pyramid in the code pass
            want0 = frame_model(g.split(src), g.planes)
            assert np.array_equal(out["frames"][k][0], want0), f"{what} lane {k}: ingested frame: {first_diff(out['frames'][k][0], want0)}"
        else:
            check_frames(port, g, k, src, out["frames"][k], what)
        luma_sum, nintra = (int(v) for v in out["misc"][k])
        if not code and p["do_sum"]:
            top = port_pyramid(port, g, src)[-1]
            assert luma_sum == int(top.astype(np.int64).sum()), f"{what} lane {k}: luma sum {luma_sum} != {int(top.sum())}"
        elif zeroed:
            assert luma_sum == 0, f"{what} lane {k}: luma sum of a lane without a sum must be zeroed, got {luma_sum}"
        if p["has_ref"] and (check is None or k in check):
            if code:
                field = mvs[k]
            else:
                pct, field = port_hme(port, g, src, lm.prev_src)
                got = out["mv"][k]
                bad = [f for f in MV_FIELDS if not np.array_equal(got[f], field[f])]
                assert not bad, f"{what} lane {k}: vector fields {bad} differ from the port's search"
                want_intra = int((field["mode"] == 1).sum())
                assert nintra == want_intra, f"{what} lane {k}: nintra {nintra} != {want_intra}"
                assert nintra * 100 // g.nblk == pct, f"{what} lane {k}: intra share {nintra * 100 // g.nblk} != {pct}"
            wp, wr = port.sub_pred(field, g.w, g.h, g.subsamp, src, lm.prev_recon, g.blk)
            assert np.array_equal(out["pred"][k], wp), f"{what} lane {k}: prediction: {first_diff(out['pred'][k], wp)}"
            assert np.array_equal(out["resid"][k], wr), f"{what} lane {k}: residual: {first_diff(out['resid'][k], wr)}"
        elif zeroed and not p["has_ref"]:
            assert nintra == 0, f"{what} lane {k}: intra count of a lane without a search must be zeroed, got {nintra}"
        lm.prev_src, lm.prev_recon = src, p["recon"]


def run_sequence(lib, port, g, schedule, seed, kinds=None, offsets=(0, 1, 3, 8), device_src=None, code_calls=1, content_fn=None,
                 check=None):
    """Calls on the same lanes: schedule[c][k] = (has_ref, do_sum) of lane k in call c of the search pass, then
    code_calls code passes with random fields (lane 0 an I picture when there are several lanes).  content_fn(k, t):
    picture t of lane k (default: `content` of kinds[k]).  Host sources are staged at the byte offsets `offsets` in
    turn; device_src(array, offset) -> (device address, keepalive) makes every other picture device-resident, read
    where it lies.  check: the lanes whose search and compensation are compared with the port (default all; the frames and
sums of every lane are checked)."""
    n = len(schedule[0])
    kinds = kinds or ["synth"] * n
    if content_fn is None:
        content_fn = lambda k, t: content(g, seed + 17 * k, t + k, kinds[k])  # noqa: E731
    check = set(range(n)) if check is None else set(check)
    me = Me(lib, g, n)
    lanes = [LaneModel() for _ in range(n)]
    rng = np.random.default_rng(seed)
    code_sched = [(0 if k == 0 and n > 1 else 1, 0) for k in range(n)]
    try:
        calls = [("search", s) for s in schedule] + [("code", code_sched)] * code_calls
        for c, (mode, sched) in enumerate(calls):
            pics, keep = [], []
            for k, (has_ref, do_sum) in enumerate(sched):
                src = content_fn(k, c)
                off = offsets[(c + k) % len(offsets)]
                p = dict(host_src=src, has_ref=has_ref, do_sum=do_sum, recon=recon_of(src, seed + 31 * c + k))
                if device_src is not None and (c + k) % 2:
                    addr, ka = device_src(src, off)
                    keep.append(ka)
                    p.update(src=addr, on_device=1)
                else:
                    p.update(src=src, stage_offset=off)
                pics.append(p)
            mvs = [random_field(rng, g.nblk) for _ in range(n)] if mode == "code" else None
            out = me.run(pics, mvs)
            check_run(port, g, lanes, pics, out, mvs, what=f"{g} call {c} ({mode})", check=check)
    finally:
        me.close()


def check_reject(lib, g):
    """a has_ref picture on a lane that has had no picture yet is refused"""
    me = Me(lib, g, 2)
    try:
        src = content(g, 1, 0)
        pics = [dict(src=src, has_ref=0, do_sum=1), dict(src=src, has_ref=1, do_sum=1)]
        me.run(pics, expect_rc=-1)
        me.run([pics[0]])  # lane 0 now has a picture, lane 1 still none
        me.run([dict(src=src, has_ref=1, do_sum=0)])
        me.run(pics, expect_rc=-1)
    finally:
        me.close()


def run_decoder(lib, port, g, isP, seed):
    """the decoder's compensation over a mix of I and P lanes: P lanes equal the port's add_pred with their own field,
    I lanes are untouched although their (unused) fields would change them"""
    rng = np.random.default_rng(seed)
    n = len(isP)
    mvs = [random_field(rng, g.nblk) for _ in range(n)]
    resid = [rng.integers(0, 256, size=g.frame_bytes, dtype=np.uint8) for _ in range(n)]
    ref = [content(g, seed + k, k, "noise" if k == 1 else "synth") for k in range(n)]
    out = add_pred_batch(lib, g, isP, mvs, resid, ref)
    for k in range(n):
        if isP[k]:
            want = port.add_pred(mvs[k], g.w, g.h, g.subsamp, resid[k], ref[k], g.blk)
            assert np.array_equal(out[k], want), f"{g} decoder lane {k} (P): {first_diff(out[k], want)}"
        else:
            assert np.array_equal(out[k], resid[k]), f"{g} decoder lane {k} (I) was written: {first_diff(out[k], resid[k])}"
