"""Host-only helpers the CLI links besides the codec (util.h: estimate_bitrate, conv444to422, conv422to420): the
library's versions against the unmodified reference's (live or recorded, tests/refdigest.py), same inputs, through
ctypes.  No GPU."""
import ctypes as C

import numpy as np

import dsvlibs as L
import refdigest


class Meta(C.Structure):
    _fields_ = [(k, C.c_int) for k in ("width", "height", "subsamp", "fps_num", "fps_den", "aspect_num", "aspect_den")]


class Plane(C.Structure):
    _fields_ = [("data", C.c_void_p), ("len", C.c_int), ("format", C.c_int), ("stride", C.c_int), ("w", C.c_int),
                ("h", C.c_int), ("hs", C.c_int), ("vs", C.c_int)]


def _bitrates(lib):
    lib = lib.lib
    lib.estimate_bitrate.restype = C.c_uint
    rng = np.random.default_rng(5)
    out = []
    for (w, h) in [(176, 144), (352, 288), (854, 480), (1920, 1080), (3840, 2160), (16, 16)]:
        for sub in L.SUBSAMP.values():
            for (fn, fd) in [(30, 1), (24, 1), (30000, 1001), (60, 1), (1, 1)]:
                for _ in range(10):
                    q, gop = int(rng.integers(0, 2048)), int(rng.integers(0, 61))
                    m = Meta(w, h, sub, fn, fd, 1, 1)
                    out.append((w, h, sub, fn, fd, q, gop, lib.estimate_bitrate(q, gop, C.byref(m))))
    return out


def test_estimate_bitrate_matches_reference(gpu, ref):
    got = _bitrates(gpu)
    assert len(got) >= 1000
    want = refdigest.table(ref, "estimate_bitrate", _bitrates)
    for a, b in zip(want, got):
        assert a == b, a[:-1]
    assert want == got


def _plane(arr, hs, vs):
    return Plane(arr.ctypes.data, arr.size, 0, arr.shape[1], arr.shape[1], arr.shape[0], hs, vs)


def _conversions(lib):
    lib = lib.lib
    rng = np.random.default_rng(6)
    outs = []
    for (w, h) in [(16, 16), (37, 21), (176, 144), (427, 240)]:
        src = rng.integers(0, 256, size=(h, w), dtype=np.uint8)
        a = np.zeros((h, (w + 1) // 2), dtype=np.uint8)
        b = np.zeros(((h + 1) // 2, (w + 1) // 2), dtype=np.uint8)
        s, d1, d2 = _plane(src, 0, 0), _plane(a, 1, 0), _plane(b, 1, 1)   # Plane holds raw pointers: no temporaries
        lib.conv444to422(C.byref(s), C.byref(d1))
        lib.conv422to420(C.byref(d1), C.byref(d2))
        outs.append((a, b))
    return outs


def test_chroma_conversions_match_reference(gpu, ref):
    got = _conversions(gpu)
    want = refdigest.table(ref, "chroma_conversions", _conversions)
    for (wa, wb), (ga, gb), wh in zip(want, got, [(16, 16), (37, 21), (176, 144), (427, 240)]):
        assert np.array_equal(wa, ga) and np.array_equal(wb, gb), wh
