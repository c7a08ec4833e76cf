"""The encoders' SSIM report (dsvb_*_picture_ssim, csrc/quality.cu) on the device at product sizes: the kernel against
the definition in numpy (picssim.plane_ssim_q32) with ==, every record against numpy's SSIM over (input, stream
decoded by dsvb_decode), streams unchanged by the report, records independent of lanes and of where the input lives,
and the recorded goldens with the report on."""
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest

import dsvlibs as L
import picinfo as PI
import picssim as PS

pytestmark = pytest.mark.gpu

GOLD = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "streams.json")))


def test_ssim_batch_gpu(gpu):
    """product sizes mixed in one launch, and one 16384-wide plane (4096 blocks per row, 32 tiles across)"""
    geos = [(1920, 1080, L.SUBSAMP["420"]), (1280, 720, L.SUBSAMP["422"]), (854, 480, L.SUBSAMP["411"]),
            (3840, 2160, L.SUBSAMP["444"]), (16384, 64, L.SUBSAMP["420"])]
    rng = np.random.default_rng(6)
    srcs, recs = [], []
    for k, (w, h, sub) in enumerate(geos):
        fb = L.frame_bytes(w, h, sub)
        a = rng.integers(0, 256, fb, dtype=np.uint8)
        if k % 2 == 0:
            a = np.sort(a)  # smooth content
        srcs.append(a)
        recs.append(np.clip(a.astype(np.int16) + rng.integers(-9, 10, fb), 0, 255).astype(np.uint8))
    recs[1] = srcs[1].copy()  # identical: exactly 2^32 per window
    sums, wins = PS.ssim_batch(gpu, geos, srcs, recs, (0, 255))
    for k, (w, h, sub) in enumerate(geos):
        assert [(int(s), int(n)) for s, n in zip(sums[k], wins[k])] == PS.plane_ssim_sums(srcs[k], recs[k], w, h, sub), k
    assert list(sums[1]) == [(1 << 32) * int(n) for n in wins[1]]
    assert list(wins[0]) == [479 * 269, 239 * 134, 239 * 134]


def encode(gpu, cfg, seqs, n, lanes, ssim, info=False, device_ptrs=None):
    be = L.BatchEncoder(gpu, cfg, lanes)
    try:
        PS.set_picture_ssim(be, ssim)
        PI.set_picture_info(be, info)
        if device_ptrs is None:
            streams = be.encode(seqs, n)
        else:
            outs = [np.zeros(len(s) + (1 << 20), dtype=np.uint8) for s in seqs]
            rc, lens = be.encode_ptrs(device_ptrs, n, 1, [o.ctypes.data for o in outs], [len(o) for o in outs])
            assert rc == 0
            streams = [o[:k].tobytes() for o, k in zip(outs, lens)]
        recs = [PS.picture_ssim(be, s) for s in range(len(seqs))]
        infos = [PI.picture_info(be, s) for s in range(len(seqs))]
    finally:
        be.close()
    return streams, recs, infos


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
    off, _, _ = encode(gpu, cfg, seqs, n, nseq, False, device_ptrs=[t.data_ptr() for t in d])
    on_dev, recs_dev, _ = encode(gpu, cfg, seqs, n, nseq, True, device_ptrs=[t.data_ptr() for t in d])
    on_host, recs_host, _ = encode(gpu, cfg, seqs, n, nseq, True)
    assert on_dev == off and on_host == off
    for s in range(nseq):
        assert recs_dev[s].tobytes() == recs_host[s].tobytes()
        PS.check_ssim(gpu, recs_dev[s], seqs[s], off[s], w, h, fmt, n)
    # the same sequences one lane at a time: identical records
    for s in (0, 1):
        one, recs_one, _ = encode(gpu, cfg, [seqs[s]], n, 1, True)
        assert one[0] == off[s] and recs_one[0].tobytes() == recs_dev[s].tobytes()


@pytest.mark.parametrize("case", [(1280, 720, "422", 4, 12, 3, 2), (854, 480, "411", 4, 12, 2, 2), (3840, 2160, "444", 2, 12, 1, 1),
                                  (1920, 1080, "420", 3, 0, 4, 4)], ids=lambda c: f"{c[0]}x{c[1]}_{c[2]}_gop{c[4]}")
def test_formats(gpu, case):
    w, h, fmt, n, gop, nseq, lanes = case
    seqs = [L.synth_sequence(w, h, fmt, n, 70 + s, 0) for s in range(nseq)]
    cfg = L.make_cfg(w, h, fmt, gop=gop)
    off, _, _ = encode(gpu, cfg, seqs, n, lanes, False)
    on, recs, _ = encode(gpu, cfg, seqs, n, lanes, True)
    assert on == off
    for s in range(nseq):
        PS.check_ssim(gpu, recs[s], seqs[s], on[s], w, h, fmt, n)


@pytest.mark.parametrize("name", ["cif_gop12", "hd_gop12"])
def test_golden_with_ssim_and_both_reports(gpu, name):
    g = GOLD[name]
    w, h, fmt, n = g["w"], g["h"], g["fmt"], g["frames"]
    yuv = L.synth_sequence(w, h, fmt, n, g["seed"], g["cut"])
    cfg = L.make_cfg(w, h, fmt, gop=g["gop"], qp=g["qp"])
    s_ssim, r_ssim, _ = encode(gpu, cfg, [yuv], n, 1, True)
    s_both, r_both, i_both = encode(gpu, cfg, [yuv], n, 1, True, info=True)
    assert hashlib.md5(s_ssim[0]).hexdigest() == g["dsv_md5"]
    assert hashlib.md5(s_both[0]).hexdigest() == g["dsv_md5"]
    assert r_both[0].tobytes() == r_ssim[0].tobytes()
    PS.check_ssim(gpu, r_ssim[0], yuv, s_ssim[0], w, h, fmt, n)
    PI.check(gpu, i_both[0], yuv, s_both[0], w, h, fmt, n)
