"""The motion kernels configured as EncEngine::step / DecEngine::step launch them, on the B200, against the plain-C port:
the cases of test_emu_motion_parity.py at full size, device-resident sources taken from CUDA tensors at byte offsets,
the bench's launch shape (64 HD lanes in one launch) and a mixed-content batch on a scene cut."""
import ctypes as C

import numpy as np
import pytest

import dsvlibs as L
import motionparity as MP
from test_emu_motion_parity import GEOMS, SCHEDULES

pytestmark = pytest.mark.gpu
ids = lambda g: f"{g[0]}x{g[1]}_{g[2]}_{'auto' if g[3] is None else '%dx%d' % g[3]}"  # noqa: E731


def device_src(a, off):
    """a CUDA tensor holding `a` at `off` bytes past a 256-byte boundary: (its address, the tensor)"""
    import torch
    t = torch.zeros(len(a) + 512, dtype=torch.uint8, device="cuda")
    base = (-t.data_ptr()) % 256
    t[base + off:base + off + len(a)] = torch.from_numpy(a).cuda()
    torch.cuda.synchronize()
    return t.data_ptr() + base + off, t


def synth(gpu, g, seed, cut=0):
    """content_fn of lanes whose pictures come from the device synthesis (bit-identical to oracle/synth.c)"""
    import torch
    cache = {}

    def fn(k, t):
        key = (k, t)
        if key not in cache:
            d = torch.empty(g.frame_bytes, dtype=torch.uint8, device="cuda")
            rc = gpu.lib.dsvb_synth_device(g.w, g.h, g.subsamp, t, 1, seed + k, cut, C.c_void_p(d.data_ptr()), 0)
            assert rc == 0, rc
            cache[key] = d.cpu().numpy()
        return cache[key]
    return fn


@pytest.mark.parametrize("geom", GEOMS, ids=ids)
def test_motion_lanes_gpu(gpu, port, geom):
    # four lanes on every geometry, lane 1 noise
    w, h, fmt, blk, _ = geom
    MP.run_sequence(gpu, port, MP.Geom(w, h, fmt, blk), SCHEDULES[4], seed=w + h, kinds=["synth", "noise", "synth", "synth"],
                    device_src=device_src)


FULL = [(1280, 720, "422", 4), (854, 480, "411", 4), (3840, 2160, "444", 2)]


@pytest.mark.parametrize("geom", FULL, ids=lambda g: f"{g[0]}x{g[1]}_{g[2]}")
def test_motion_full_size_gpu(gpu, port, geom):
    w, h, fmt, n = geom
    g = MP.Geom(w, h, fmt)
    MP.run_sequence(gpu, port, g, SCHEDULES[n], seed=w, device_src=device_src, content_fn=synth(gpu, g, w))


def test_motion_bench_shape_gpu(gpu, port):
    """64 HD 4:2:0 lanes in one launch (the bench's batch): every lane is checked against the frame model, one lane in
    eight (first and last included) against the port's search and compensation.  Lanes differ: each shifts one
    synthetic sequence by its own offset, and lane 5 is noise."""
    g = MP.Geom(1920, 1080, "420")
    n = 64
    base = synth(gpu, g, 7)
    rng = np.random.default_rng(64)
    shifts = [(int(rng.integers(-40, 41)), int(rng.integers(-40, 41))) for _ in range(n)]

    def content(k, t):
        if k == 5:
            return MP.content(g, 99, t, "noise")
        planes = g.split(base(0, t))
        return np.concatenate([np.roll(p, (shifts[k][0] >> (p.shape[0] != g.h), shifts[k][1] >> (p.shape[1] != g.w)),
                                       axis=(0, 1)).ravel() for p in planes])
    schedule = [[(0, 1)] * n, [(k % 7 != 3, k % 3 != 1) for k in range(n)], [(k % 5 != 0, 1) for k in range(n)]]
    MP.run_sequence(gpu, port, g, schedule, seed=7, device_src=device_src, content_fn=content,
                    check={k for k in range(n) if k % 8 == 0 or k in (5, 63)})


def test_motion_scene_cut_gpu(gpu, port):
    """a batch of mixed content on a scene cut: HD lanes of four sequences, two of which cut at their third picture"""
    g = MP.Geom(1920, 1080, "420")
    cut = synth(gpu, g, 11, cut=2)
    plain = synth(gpu, g, 21)
    MP.run_sequence(gpu, port, g, SCHEDULES[4], seed=11, device_src=device_src,
                    content_fn=lambda k, t: (cut if k % 2 == 0 else plain)(k, t))


@pytest.mark.parametrize("geom", GEOMS + [(1920, 1080, "420", None, 0), (854, 480, "411", None, 0)], ids=ids)
def test_decoder_compensation_gpu(gpu, port, geom):
    w, h, fmt, blk, _ = geom
    MP.run_decoder(gpu, port, MP.Geom(w, h, fmt, blk), isP=[0, 1, 1, 0, 1, 1], seed=w * h)


def test_motion_reject_gpu(gpu):
    MP.check_reject(gpu, MP.Geom(54, 38, "420"))
