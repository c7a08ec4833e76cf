"""The encoders' SSIM report (dsvb_*_picture_ssim, include/dsv1_b200_batch.h) from Python, and checks of it.

Bindings: set_picture_ssim / picture_ssim take a dsvlibs.BatchEncoder or dsvlibs.MultiGpu and return numpy records of
PICSSIM_DTYPE; ssim_batch calls the kernel-level dsvk_ssim_batch.  plane_ssim_q32 is the definition at DSVB_PICSSIM
in numpy, and check_ssim compares records with it over (input, stream decoded by dsvb_decode).  Used by
test_emu_picture_ssim.py (CPU emulation), test_gpu_picture_ssim.py (B200) and tools/picture_info_cost.py --report ssim."""
import ctypes as C

import numpy as np

import dsvlibs as L
from picinfo import decode


# DSVB_PICSSIM: one coded picture of the SSIM report
PICSSIM_DTYPE = np.dtype([("ssim", "<f8", (3,)), ("windows", "<i8", (3,))])
assert PICSSIM_DTYPE.itemsize == 48


def _ssim_api(obj):
    if isinstance(obj, L.MultiGpu):
        return obj.lib.dsvb_multi_set_picture_ssim, obj.lib.dsvb_multi_picture_ssim
    return obj.lib.dsvb_enc_set_picture_ssim, obj.lib.dsvb_enc_picture_ssim


def set_picture_ssim(obj, on):
    _ssim_api(obj)[0](obj.h, int(on))


def picture_ssim(obj, seq=0):
    """PICSSIM_DTYPE records of sequence seq of the last encode call, in picture order; None where the library
    returns -1"""
    fn = _ssim_api(obj)[1]
    n = fn(obj.h, int(seq), None, 0)
    if n < 0:
        return None
    out = np.zeros(n, dtype=PICSSIM_DTYPE)
    got = fn(obj.h, int(seq), out.ctypes.data_as(C.c_void_p), n)
    assert got == n, (got, n)
    return out


def ssim_batch(lib, geos, srcs, recs, fill=(0, 255)):
    """dsvk_ssim_batch, arguments as sse_batch.  Returns ((n, 3) int64 window sums, (n, 3) int64 window counts)."""
    n = len(geos)
    geo = np.array([v for g in geos for v in g], dtype=np.int32)
    src = np.ascontiguousarray(np.concatenate(srcs), dtype=np.uint8)
    rec = np.ascontiguousarray(np.concatenate(recs), dtype=np.uint8)
    bf = np.array(fill, dtype=np.uint8)
    sums = np.zeros((n, 3), dtype=np.int64)
    wins = np.zeros((n, 3), dtype=np.int64)
    rc = lib.lib.dsvk_ssim_batch(n, L.ptr(geo, L.i32p), L.ptr(src), L.ptr(rec), L.ptr(bf), sums.ctypes.data_as(C.c_void_p),
                                 wins.ctypes.data_as(C.c_void_p))
    assert rc == 0, rc
    return sums, wins


SSIM_C1, SSIM_C2 = 416, 235963  # x264's ssim_c1 / ssim_c2 for 8-bit samples


def plane_ssim_q32(a, b):
    """the definition at DSVB_PICSSIM: a, b (ph, pw) uint8 -> (sum over windows of rint(ssim_w * 2^32), windows)"""
    ph, pw = a.shape
    bw, bh = pw // 4, ph // 4
    if bw < 2 or bh < 2:
        return 0, 0
    a = a[:4 * bh, :4 * bw].astype(np.int64)
    b = b[:4 * bh, :4 * bw].astype(np.int64)

    def blk(x):
        return x.reshape(bh, 4, bw, 4).sum(axis=(1, 3))

    def win(x):
        return x[:-1, :-1] + x[1:, :-1] + x[:-1, 1:] + x[1:, 1:]

    s1, s2, ss, s12 = (win(blk(x)) for x in (a, b, a * a + b * b, a * b))
    vars_ = 64 * ss - s1 * s1 - s2 * s2
    covar = 64 * s12 - s1 * s2
    num = (2 * s1 * s2 + SSIM_C1) * (2 * covar + SSIM_C2)
    den = (s1 * s1 + s2 * s2 + SSIM_C1) * (vars_ + SSIM_C2)
    q = np.rint(num.astype(np.float64) / den.astype(np.float64) * 4294967296.0).astype(np.int64)
    return int(q.sum()), int(q.size)


def plane_ssim_sums(a, b, w, h, sub):
    """[(S, windows)] per plane of two packed frames"""
    out, off = [], 0
    for pw, ph in L.plane_dims(w, h, sub):
        out.append(plane_ssim_q32(a[off:off + pw * ph].reshape(ph, pw), b[off:off + pw * ph].reshape(ph, pw)))
        off += pw * ph
    return out


def ssim_value(s, windows):
    """the reported value: S / 2^32 / windows, NaN without windows"""
    return float(s) / 4294967296.0 / float(windows) if windows else float("nan")


def check_ssim(lib, recs, yuv, stream, w, h, fmt, n, dec=None):
    """every record == numpy's SSIM over (input picture k, picture k of the stream decoded by dsvb_decode); returns
    the decoded pictures"""
    sub = L.SUBSAMP[fmt]
    fb = L.frame_bytes(w, h, sub)
    assert recs is not None and len(recs) == n
    if dec is None:
        dec = decode(lib, stream, w, h, sub, n)
    for f, r in enumerate(recs):
        want = plane_ssim_sums(yuv[f * fb:(f + 1) * fb], dec[f * fb:(f + 1) * fb], w, h, sub)
        assert [int(v) for v in r["windows"]] == [wn for _, wn in want], (f, list(r["windows"]), want)
        for p, (s, wn) in enumerate(want):
            v = ssim_value(s, wn)
            assert (np.isnan(v) and np.isnan(r["ssim"][p])) or float(r["ssim"][p]) == v, (f, p, float(r["ssim"][p]), v)
    return dec
