"""The encoders' SSIM report (dsvb_*_picture_ssim, csrc/quality.cu) on the test-only CPU emulation of the CUDA sources:
the SSIM kernel through dsvk_ssim_batch against the definition in numpy (picssim.plane_ssim_q32), compared with ==,
and whole encodes with the report on against the streams they produce.  Small sizes; test_gpu_picture_ssim.py runs
product sizes on the device."""
import subprocess

import numpy as np
import pytest

import dsvlibs as L
import picinfo as PI
import picssim as PS

Q32 = 1 << 32


@pytest.fixture(scope="module")
def emu():
    subprocess.run(["make", "-s", "-C", L.PKG, "emu"], check=True, stdout=subprocess.DEVNULL)
    return L.emu()


def ssim_case(lib, geos, seed, fills):
    rng = np.random.default_rng(seed)
    srcs, recs = [], []
    for i, (w, h, sub) in enumerate(geos):
        fb = L.frame_bytes(w, h, sub)
        a = rng.integers(0, 256, fb, dtype=np.uint8)
        if i % 4 == 0:  # smooth content: values near 1
            a = np.sort(a)
        b = np.clip(a.astype(np.int16) + rng.integers(-20, 21, fb), 0, 255).astype(np.uint8)
        srcs.append(a)
        recs.append(b)
    sums, wins = PS.ssim_batch(lib, geos, srcs, recs, fills)
    for k, (w, h, sub) in enumerate(geos):
        want = PS.plane_ssim_sums(srcs[k], recs[k], w, h, sub)
        assert [(int(s), int(n)) for s, n in zip(sums[k], wins[k])] == want, (k, w, h, sub)
    return sums, wins


SUBS = [L.SUBSAMP[f] for f in ("420", "411", "422", "444")]


def test_ssim_batch_widths_emu(emu):
    """every even width 16..34 over all four chroma formats, heights 16..26 (luma and chroma sizes with % 4 != 0),
    mixed in one launch; border / padding bytes that differ between the frames, both ways round"""
    geos = [(w, 16 + (w % 12), SUBS[i % 4]) for i, w in enumerate(range(16, 36, 2))]
    ssim_case(emu, geos, 1, (0, 255))
    ssim_case(emu, geos[::-1], 2, (255, 0))


def test_ssim_batch_411_edges_emu(emu):
    """4:1:1 chroma narrower than 8 samples (widths 16..28) has no windows; width 30 gives chroma 8 wide: one window
    column"""
    geos = [(w, 22, L.SUBSAMP["411"]) for w in range(16, 32, 2)]
    sums, wins = ssim_case(emu, geos, 3, (0, 255))
    assert (wins[:-1, 1:] == 0).all() and (sums[:-1, 1:] == 0).all()
    assert list(wins[-1]) == [(30 // 4 - 1) * 4, 4, 4]


def test_ssim_batch_multi_tile_emu(emu):
    """a plane larger than one CTA tile (128 x 14 windows) in both directions, beside a small one"""
    ssim_case(emu, [(520, 200, L.SUBSAMP["444"]), (18, 34, L.SUBSAMP["420"])], 4, (255, 0))


def test_ssim_special_inputs_emu(emu):
    w, h, sub = 64, 40, L.SUBSAMP["420"]
    fb = L.frame_bytes(w, h, sub)
    x = np.random.default_rng(5).integers(0, 256, fb, dtype=np.uint8)
    zero, full = np.zeros(fb, np.uint8), np.full(fb, 255, np.uint8)
    sums, wins = PS.ssim_batch(emu, [(w, h, sub)] * 4, [x, x, zero, x], [x, x[::-1].copy(), full, 255 - x], (0, 255))
    assert list(sums[0]) == [Q32 * n for n in wins[0]]  # identical planes: exactly 1 per window
    assert list(wins[0]) == [15 * 9, 7 * 4, 7 * 4]
    for k in (1, 2, 3):
        want = PS.plane_ssim_sums([x, x, zero, x][k], [x, x[::-1], full, 255 - x][k], w, h, sub)
        assert [(int(s), int(n)) for s, n in zip(sums[k], wins[k])] == want
    assert (sums[3] < 0).all()  # 255 - x: negative correlation
    assert (sums[2] > 0).all() and (sums[2] < wins[2] * Q32 // 1000).all()  # 0 against 255: near 0


def test_ssim_batch_rejects_illegal_geometry_emu(emu):
    geo = np.array([15, 16, L.SUBSAMP["420"]], dtype=np.int32)
    buf = np.zeros(1024, np.uint8)
    out = np.zeros(3, np.int64)
    rc = emu.lib.dsvk_ssim_batch(1, L.ptr(geo, L.i32p), L.ptr(buf), L.ptr(buf), L.ptr(np.zeros(2, np.uint8)),
                                 out.ctypes.data_as(PS.C.c_void_p), out.ctypes.data_as(PS.C.c_void_p))
    assert rc == -1


# launch counts of the same calls with no report on (test_emu_picture_info.py)
LAUNCHES_OFF = {"gop12": 198, "gop0": 56}


def batch(lib, w, h, fmt, n, nseq, lanes, seed, cut, info, ssim, **kw):
    cfg = L.make_cfg(w, h, fmt, **kw)
    seqs = [L.synth_sequence(w, h, fmt, n, seed + s, cut) for s in range(nseq)]
    be = L.BatchEncoder(lib, cfg, lanes)
    try:
        PI.set_picture_info(be, info)
        PS.set_picture_ssim(be, ssim)
        streams = be.encode(seqs, n)
        infos = [PI.picture_info(be, s) for s in range(nseq)]
        ssims = [PS.picture_ssim(be, s) for s in range(nseq)]
        assert PS.picture_ssim(be, nseq) is None and PS.picture_ssim(be, -1) is None
        launches = be.stats()["kernel_launches"]
    finally:
        be.close()
    return seqs, streams, infos, ssims, launches


@pytest.mark.parametrize("case", [
    # name, w, h, fmt, frames, sequences, lanes, seed, cut, cfg; extra launches per step with only the SSIM report on
    ("gop12", 32, 32, "420", 5, 3, 2, 3, 3, dict(gop=12), 1),          # scene cut: a forced I picture; 3 sequences on 2 lanes
    ("gop0", 32, 32, "420", 4, 3, 2, 3, 0, dict(gop=0), 4),            # intra only: the inverse runs only for the report
    ("444", 48, 32, "444", 3, 1, 1, 5, 0, dict(gop=12), 1),
    ("411", 36, 34, "411", 3, 2, 2, 6, 0, dict(gop=2), 1),             # chroma 9 x 34: one window column
    ("411_narrow", 28, 32, "411", 3, 1, 1, 9, 0, dict(gop=12), 1),     # chroma 7 wide: no windows, NaN
    ("abr", 32, 32, "420", 8, 1, 1, 7, 0, dict(gop=12, rc_mode=1, bitrate=20000, quality=L.qp_to_quality(60)), 1),
    ("refresh", 32, 32, "420", 6, 1, 1, 8, 0, dict(gop=6, stable_refresh=2), 1),
], ids=lambda c: c[0])
def test_batch_picture_ssim_emu(emu, case):
    name, w, h, fmt, n, nseq, lanes, seed, cut, kw, per_step = case
    steps = n * ((nseq + lanes - 1) // lanes)
    _, s_off, i_off, r_off, l_off = batch(emu, w, h, fmt, n, nseq, lanes, seed, cut, False, False, **kw)
    assert r_off == [None] * nseq and i_off == [None] * nseq  # both reports were off
    if name in LAUNCHES_OFF:
        assert l_off == LAUNCHES_OFF[name]
    seqs, s_on, i_on, recs, l_on = batch(emu, w, h, fmt, n, nseq, lanes, seed, cut, False, True, **kw)
    assert s_on == s_off
    assert i_on == [None] * nseq  # the SSE report stays off
    assert l_on == l_off + per_step * steps
    _, s_sse, i_sse, r_sse, l_sse = batch(emu, w, h, fmt, n, nseq, lanes, seed, cut, True, False, **kw)
    _, s_both, i_both, r_both, l_both = batch(emu, w, h, fmt, n, nseq, lanes, seed, cut, True, True, **kw)
    assert s_sse == s_off and s_both == s_off
    assert r_sse == [None] * nseq
    assert l_both == l_sse + steps  # the second report adds its kernel only
    for s in range(nseq):
        assert np.array_equal(i_both[s], i_sse[s])  # DSVB_PICINFO unchanged by the SSIM report
        assert r_both[s].tobytes() == recs[s].tobytes()
        PS.check_ssim(emu, recs[s], seqs[s], s_on[s], w, h, fmt, n)
    allr = np.concatenate(recs)
    if name == "411_narrow":
        assert (allr["windows"][:, 1:] == 0).all() and np.isnan(allr["ssim"][:, 1:]).all()
    else:
        assert (allr["windows"] > 0).all() and (allr["ssim"] < 1).any()


def test_encode_long_picture_ssim_emu(emu):
    """dsvb_encode_long over 2 lanes (chains out of order on the lanes, a forced I picture at the cut) and MultiGpu over
    two emulated devices give the records of a one-lane dsvb_encode of the same sequence"""
    w, h, fmt, n = 32, 32, "420", 7
    fb = L.frame_bytes(w, h, L.SUBSAMP[fmt])
    yuv = L.synth_sequence(w, h, fmt, n, 7, 4)
    cfg = L.make_cfg(w, h, fmt, gop=3, qp=70, stable_refresh=2)
    one = L.BatchEncoder(emu, cfg, 1)
    PS.set_picture_ssim(one, 1)
    want_stream = one.encode([yuv], n)[0]
    want = PS.picture_ssim(one, 0)
    one.close()
    PS.check_ssim(emu, want, yuv, want_stream, w, h, fmt, n)

    be = L.BatchEncoder(emu, cfg, 2)
    be.encode_long(yuv, n)
    assert PS.picture_ssim(be, 0) is None
    PS.set_picture_ssim(be, 1)
    got, info = be.encode_long(yuv, n)
    assert info[1] == 1
    assert PS.picture_ssim(be, 0).tobytes() == want.tobytes()
    assert PS.picture_ssim(be, 1) is None and PI.picture_info(be, 0) is None
    PS.set_picture_ssim(be, 0)
    be.encode_long(yuv, n)
    assert PS.picture_ssim(be, 0) is None
    be.close()

    mg = L.MultiGpu(emu, cfg, 1, [0, 0])
    PS.set_picture_ssim(mg, 1)
    got, info = mg.encode_long(yuv, n)
    assert info[3] == 2
    assert PS.picture_ssim(mg, 0).tobytes() == want.tobytes()
    seqs = [yuv[:fb * 4]] + [L.synth_sequence(w, h, fmt, 4, 20 + s, 0) for s in range(2)]
    streams = mg.encode(seqs, 4)
    assert PS.picture_ssim(mg, 0).tobytes() == want[:4].tobytes()
    for s in range(3):
        PS.check_ssim(emu, PS.picture_ssim(mg, s), seqs[s], streams[s], w, h, fmt, 4)
    assert PS.picture_ssim(mg, 3) is None and PI.picture_info(mg, 0) is None
    mg.close()
