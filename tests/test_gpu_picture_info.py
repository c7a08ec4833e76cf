"""The encoders' per-picture report (dsvb_*_picture_info, csrc/quality.cu) on the device at product sizes: every record
against the stream it describes and numpy's squared error over (input, stream decoded by dsvb_decode) (picinfo.py),
streams unchanged by the report, and the recorded goldens with the report on."""
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest

import dsvlibs as L
import picinfo as PI

pytestmark = pytest.mark.gpu

GOLD = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "streams.json")))


def test_sse_batch_gpu(gpu):
    """the kernel through dsvk_sse_batch at product sizes, mixed formats in one launch, 0 against 255 over a whole UHD
    plane (5.4e11, past 32 bits)"""
    geos = [(1920, 1080, L.SUBSAMP["420"]), (854, 480, L.SUBSAMP["411"]), (1280, 720, L.SUBSAMP["422"]),
            (3840, 2160, L.SUBSAMP["444"]), (34, 18, L.SUBSAMP["420"])]
    rng = np.random.default_rng(5)
    srcs, recs = [], []
    for w, h, sub in geos:
        fb = L.frame_bytes(w, h, sub)
        a = rng.integers(0, 256, fb, dtype=np.uint8)
        srcs.append(a)
        recs.append(np.clip(a.astype(np.int16) + rng.integers(-9, 10, fb), 0, 255).astype(np.uint8))
    srcs[3] = np.zeros_like(srcs[3])
    recs[3] = np.full_like(recs[3], 255)
    got = PI.sse_batch(gpu, geos, srcs, recs, (0, 255))
    for k, (w, h, sub) in enumerate(geos):
        assert [int(v) for v in got[k]] == PI.plane_sse(srcs[k], recs[k], w, h, sub), k
    assert int(got[3][0]) == 3840 * 2160 * 255 ** 2


def encode(gpu, cfg, seqs, n, lanes, on, device_ptrs=None):
    be = L.BatchEncoder(gpu, cfg, lanes)
    try:
        if on:
            PI.set_picture_info(be, 1)
        if device_ptrs is None:
            streams = be.encode(seqs, n)
        else:
            outs = [np.zeros(len(s) + (1 << 20), dtype=np.uint8) for s in seqs]
            rc, lens = be.encode_ptrs(device_ptrs, n, 1, [o.ctypes.data for o in outs], [len(o) for o in outs])
            assert rc == 0
            streams = [o[:k].tobytes() for o, k in zip(outs, lens)]
        recs = [PI.picture_info(be, s) for s in range(len(seqs))]
    finally:
        be.close()
    return streams, recs


def test_hd_gop12_16_lanes_device_and_host(gpu):
    import torch
    w, h, fmt, n, nseq = 1920, 1080, "420", 12, 16
    sub = L.SUBSAMP[fmt]
    fb = L.frame_bytes(w, h, sub)
    d = [torch.zeros(fb * n, dtype=torch.uint8, device="cuda") for _ in range(nseq)]
    for s in range(nseq):
        gpu.lib.dsvb_synth_device(w, h, sub, 0, n, 60 + s, 6 if s % 4 == 1 else 0, C.c_void_p(d[s].data_ptr()), 0)
    seqs = [t.cpu().numpy() for t in d]
    cfg = L.make_cfg(w, h, fmt, gop=12)
    off, _ = encode(gpu, cfg, seqs, n, nseq, False, [t.data_ptr() for t in d])
    on_dev, recs_dev = encode(gpu, cfg, seqs, n, nseq, True, [t.data_ptr() for t in d])
    on_host, recs_host = encode(gpu, cfg, seqs, n, nseq, True)
    assert on_dev == off and on_host == off
    for s in range(nseq):
        assert np.array_equal(recs_dev[s], recs_host[s])
        PI.check(gpu, recs_dev[s], seqs[s], off[s], w, h, fmt, n)
    assert sum(int(r["forced_intra"].sum()) for r in recs_dev) > 0


@pytest.mark.parametrize("case", [(1280, 720, "422", 4, 12, 3, 2), (854, 480, "411", 4, 12, 2, 2), (3840, 2160, "444", 2, 12, 1, 1),
                                  (1920, 1080, "420", 3, 0, 4, 4)], ids=lambda c: f"{c[0]}x{c[1]}_{c[2]}_gop{c[4]}")
def test_formats(gpu, case):
    w, h, fmt, n, gop, nseq, lanes = case
    seqs = [L.synth_sequence(w, h, fmt, n, 70 + s, 0) for s in range(nseq)]
    cfg = L.make_cfg(w, h, fmt, gop=gop)
    off, _ = encode(gpu, cfg, seqs, n, lanes, False)
    on, recs = encode(gpu, cfg, seqs, n, lanes, True)
    assert on == off
    for s in range(nseq):
        PI.check(gpu, recs[s], seqs[s], on[s], w, h, fmt, n, inter=gop != 0)


def test_cif_golden_encode_long_4_lanes(gpu):
    g = GOLD["cif_gop12"]
    w, h, fmt, n = g["w"], g["h"], g["fmt"], g["frames"]
    yuv = L.synth_sequence(w, h, fmt, n, g["seed"], g["cut"])
    be = L.BatchEncoder(gpu, L.make_cfg(w, h, fmt, gop=g["gop"], qp=g["qp"]), 4)
    PI.set_picture_info(be, 1)
    stream, info = be.encode_long(yuv, n)
    recs = PI.picture_info(be, 0)
    be.close()
    assert hashlib.md5(stream).hexdigest() == g["dsv_md5"]
    PI.check(gpu, recs, yuv, stream, w, h, fmt, n)
    assert int(recs["forced_intra"].sum()) == info[1] == 1


def test_hd_gop12_golden_with_report(gpu):
    g = GOLD["hd_gop12"]
    w, h, fmt, n = g["w"], g["h"], g["fmt"], g["frames"]
    yuv = L.synth_sequence(w, h, fmt, n, g["seed"], g["cut"])
    streams, recs = encode(gpu, L.make_cfg(w, h, fmt, gop=g["gop"], qp=g["qp"]), [yuv], n, 1, True)
    assert hashlib.md5(streams[0]).hexdigest() == g["dsv_md5"]
    PI.check(gpu, recs[0], yuv, streams[0], w, h, fmt, n)
