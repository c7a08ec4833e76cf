"""The encoders' per-picture report (dsvb_*_picture_info, csrc/quality.cu) on the test-only CPU emulation of the CUDA
sources: the squared-error kernel through dsvk_sse_batch against numpy, and whole encodes with the report on against
the streams they produce (picinfo.py).  Small sizes; test_gpu_picture_info.py runs product sizes on the device."""
import subprocess

import numpy as np
import pytest

import dsvlibs as L
import picinfo as PI


@pytest.fixture(scope="module")
def emu():
    subprocess.run(["make", "-s", "-C", L.PKG, "emu"], check=True, stdout=subprocess.DEVNULL)
    return L.emu()


def sse_case(lib, geos, seed, fills):
    rng = np.random.default_rng(seed)
    srcs, recs = [], []
    for i, (w, h, sub) in enumerate(geos):
        fb = L.frame_bytes(w, h, sub)
        if i % 3 == 0:  # extremes: every sample 0 against 255
            a, b = np.zeros(fb, np.uint8), np.full(fb, 255, np.uint8)
        else:
            a = rng.integers(0, 256, fb, dtype=np.uint8)
            b = np.clip(a.astype(np.int16) + rng.integers(-40, 41, fb), 0, 255).astype(np.uint8)
        srcs.append(a)
        recs.append(b)
    got = PI.sse_batch(lib, geos, srcs, recs, fills)
    for k, (w, h, sub) in enumerate(geos):
        assert [int(v) for v in got[k]] == PI.plane_sse(srcs[k], recs[k], w, h, sub), (k, w, h, sub)


def test_sse_batch_emu(emu):
    """every even width 16..32 over all four chroma formats (odd chroma widths: 4:1:1 rows of 5, 7, 9 samples; 4:2:0 / 4:2:2
    rows of 9, 11, 13, 15), 36x32 4:1:1 (9-sample chroma rows), mixed formats in one call, and border / padding bytes
    that differ between the two frames, both ways round"""
    subs = [L.SUBSAMP[f] for f in ("420", "411", "422", "444")]
    geos = [(w, 16 + (w % 6), subs[i % 4]) for i, w in enumerate(range(16, 34, 2))] + [(36, 32, L.SUBSAMP["411"])]
    sse_case(emu, geos, 1, (0, 255))
    sse_case(emu, geos[::-1], 2, (255, 0))
    sse_case(emu, [(34, 18, L.SUBSAMP["420"]), (16, 16, L.SUBSAMP["444"])], 3, (7, 200))


# launch counts of the same calls with the report never turned on, measured at the commit before it existed
LAUNCHES_OFF = {"gop12": 198, "gop0": 56}


def batch(lib, w, h, fmt, n, nseq, lanes, seed, cut, on, **kw):
    cfg = L.make_cfg(w, h, fmt, **kw)
    seqs = [L.synth_sequence(w, h, fmt, n, seed + s, cut) for s in range(nseq)]
    be = L.BatchEncoder(lib, cfg, lanes)
    try:
        if on:
            PI.set_picture_info(be, 1)
        streams = be.encode(seqs, n)
        recs = [PI.picture_info(be, s) for s in range(nseq)]
        assert PI.picture_info(be, nseq) is None and PI.picture_info(be, -1) is None
        launches = be.stats()["kernel_launches"]
    finally:
        be.close()
    return seqs, streams, recs, launches


@pytest.mark.parametrize("case", [
    # name, w, h, fmt, frames, sequences, lanes, seed, cut, cfg; extra launches per step with the report on
    ("gop12", 32, 32, "420", 5, 3, 2, 3, 3, dict(gop=12), 1),          # scene cut: a forced I picture; 3 sequences on 2 lanes
    ("gop0", 32, 32, "420", 4, 3, 2, 3, 0, dict(gop=0), 4),            # intra only: the inverse runs only for the report
    ("444", 48, 32, "444", 3, 1, 1, 5, 0, dict(gop=12), 1),
    ("411", 36, 32, "411", 3, 2, 2, 6, 0, dict(gop=2), 1),             # 9-sample chroma rows
    ("abr", 32, 32, "420", 8, 1, 1, 7, 0, dict(gop=12, rc_mode=1, bitrate=20000, quality=L.qp_to_quality(60)), 1),
    ("refresh", 32, 32, "420", 6, 1, 1, 8, 0, dict(gop=6, stable_refresh=2), 1),
], ids=lambda c: c[0])
def test_batch_picture_info_emu(emu, case):
    name, w, h, fmt, n, nseq, lanes, seed, cut, kw, per_step = case
    _, s_off, r_off, l_off = batch(emu, w, h, fmt, n, nseq, lanes, seed, cut, False, **kw)
    assert r_off == [None] * nseq  # the report was off
    seqs, s_on, recs, l_on = batch(emu, w, h, fmt, n, nseq, lanes, seed, cut, True, **kw)
    assert s_on == s_off
    steps = n * ((nseq + lanes - 1) // lanes)
    assert l_on == l_off + per_step * steps
    if name in LAUNCHES_OFF:
        assert l_off == LAUNCHES_OFF[name]
    for s in range(nseq):
        PI.check(emu, recs[s], seqs[s], s_on[s], w, h, fmt, n, inter=kw["gop"] != 0)
    allr = np.concatenate(recs)
    if name == "gop12":
        assert allr["forced_intra"].sum() > 0 and allr["is_p"].sum() > 0
    if name == "gop0":
        assert allr["is_p"].sum() == 0
    if name == "abr":
        assert len(set(allr["quant"].tolist())) > 1


def test_encode_long_picture_info_emu(emu):
    """dsvb_encode_long over 2 lanes (chains out of order on the lanes, a forced I picture at the cut), then the same
    sequence through MultiGpu over two emulated devices, single sequences and whole ones"""
    w, h, fmt, n = 32, 32, "420", 7
    fb = L.frame_bytes(w, h, L.SUBSAMP[fmt])
    yuv = L.synth_sequence(w, h, fmt, n, 7, 4)
    cfg = L.make_cfg(w, h, fmt, gop=3, qp=70, stable_refresh=2)
    be = L.BatchEncoder(emu, cfg, 2)
    want, _ = be.encode_long(yuv, n)
    assert PI.picture_info(be, 0) is None
    PI.set_picture_info(be, 1)
    got, info = be.encode_long(yuv, n)
    recs = PI.picture_info(be, 0)
    assert PI.picture_info(be, 1) is None
    PI.set_picture_info(be, 0)
    be.encode_long(yuv, n)
    assert PI.picture_info(be, 0) is None
    be.close()
    assert got == want and info[1] == 1
    PI.check(emu, recs, yuv, got, w, h, fmt, n)
    assert recs["forced_intra"].sum() == 1

    mg = L.MultiGpu(emu, cfg, 1, [0, 0])
    PI.set_picture_info(mg, 1)
    got, info = mg.encode_long(yuv[:fb * 5], 5)
    assert info[3] == 2
    PI.check(emu, PI.picture_info(mg, 0), yuv[:fb * 5], got, w, h, fmt, 5)
    seqs = [L.synth_sequence(w, h, fmt, 4, 20 + s, 0) for s in range(3)]
    streams = mg.encode(seqs, 4)
    for s in range(3):
        PI.check(emu, PI.picture_info(mg, s), seqs[s], streams[s], w, h, fmt, 4)
    assert PI.picture_info(mg, 3) is None
    mg.close()
