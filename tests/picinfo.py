"""The encoders' per-picture report (dsvb_*_picture_info, include/dsv1_b200_batch.h) from Python, and checks of it.

Bindings: set_picture_info / picture_info take a dsvlibs.BatchEncoder or dsvlibs.MultiGpu and return numpy records of
PICINFO_DTYPE; sse_batch calls the kernel-level dsvk_sse_batch.

Checks: every record against the stream it describes -- the packets walked by their next links and type bytes, their
heads parsed up to the quantiser -- and the squared error recomputed in numpy from the input and the stream decoded by
dsvb_decode.  Used by test_emu_picture_info.py (CPU emulation), test_gpu_picture_info.py (B200) and
tools/picture_info_cost.py."""
import ctypes as C

import numpy as np

import dsvlibs as L

# DSVB_PICINFO: one coded picture of the report
PICINFO_DTYPE = np.dtype([("sse", "<u8", (3,)), ("samples", "<i8", (3,)), ("fnum", "<i8"), ("is_p", "<i4"),
                          ("forced_intra", "<i4"), ("quant", "<i4"), ("bytes", "<i4")])
assert PICINFO_DTYPE.itemsize == 72


def _api(obj):
    """(set, get) entry points of a BatchEncoder or a MultiGpu"""
    if isinstance(obj, L.MultiGpu):
        return obj.lib.dsvb_multi_set_picture_info, obj.lib.dsvb_multi_picture_info
    return obj.lib.dsvb_enc_set_picture_info, obj.lib.dsvb_enc_picture_info


def set_picture_info(obj, on):
    _api(obj)[0](obj.h, int(on))


def picture_info(obj, seq=0):
    """PICINFO_DTYPE records of sequence seq of the last encode call (seq 0 for encode_long), in picture order; None
    where the library returns -1 (report off during that call, the call failed, seq out of range)"""
    fn = _api(obj)[1]
    n = fn(obj.h, int(seq), None, 0)
    if n < 0:
        return None
    out = np.zeros(n, dtype=PICINFO_DTYPE)
    got = fn(obj.h, int(seq), out.ctypes.data_as(C.c_void_p), n)
    assert got == n, (got, n)
    return out


def psnr(sse, samples):
    """10 log10(255^2 * samples / sse) per element; inf where sse == 0"""
    sse = np.asarray(sse, dtype=np.float64)
    with np.errstate(divide="ignore"):
        return 10 * np.log10(255.0 ** 2 * np.asarray(samples, dtype=np.float64) / sse)


def sse_batch(lib, geos, srcs, recs, fill=(0, 255)):
    """dsvk_sse_batch: geos [(w, h, subsamp)], srcs / recs packed frames; border and padding bytes of the device frames
    set to fill[0] (src) and fill[1] (rec).  Returns (n, 3) uint64 sums."""
    n = len(geos)
    geo = np.array([v for g in geos for v in g], dtype=np.int32)
    src = np.ascontiguousarray(np.concatenate(srcs), dtype=np.uint8)
    rec = np.ascontiguousarray(np.concatenate(recs), dtype=np.uint8)
    bf = np.array(fill, dtype=np.uint8)
    out = np.zeros((n, 3), dtype=np.uint64)
    rc = lib.lib.dsvk_sse_batch(n, L.ptr(geo, L.i32p), L.ptr(src), L.ptr(rec), L.ptr(bf), out.ctypes.data_as(C.c_void_p))
    assert rc == 0, rc
    return out

HDR = 14          # DSV_PACKET_HDR_SIZE
PT_META, PT_EOS = 0x00, 0x10
QP_BITS = 11      # DSV_MAX_QP_BITS


class Bits:
    def __init__(self, b, byte_pos):
        self.b, self.pos = b, byte_pos * 8

    def bit(self):
        v = (int(self.b[self.pos >> 3]) >> (7 - (self.pos & 7))) & 1
        self.pos += 1
        return v

    def bits(self, n):
        v = 0
        for _ in range(n):
            v = (v << 1) | self.bit()
        return v

    def ueg(self):  # interleaved exp-Golomb: (0, bit)* then 1
        x = 1
        while not self.bit():
            x = (x << 1) | self.bit()
        return x - 1

    def align(self):
        self.pos = (self.pos + 7) & ~7

    def skip(self, nbytes):
        self.pos += 8 * nbytes


def walk(stream):
    """[(type, size, fnum, quant, after_meta)] of the picture packets, plus the bytes of all other packets"""
    b = np.frombuffer(stream, dtype=np.uint8)
    at, pics, other, prev_type = 0, [], 0, None
    while at + HDR <= len(b):
        assert bytes(b[at:at + 4]) == b"DSV1"
        t = int(b[at + 5])
        size = int.from_bytes(bytes(b[at + 10:at + 14]), "big") or HDR
        if t & 0x4:
            r = Bits(b, at + HDR)
            fnum = r.bits(32)
            r.align()
            r.ueg()
            r.ueg()
            r.align()
            r.align()
            r.skip(r.ueg())  # stability map
            if t & 1:
                for _ in range(4):  # motion sub-streams
                    r.align()
                    n = r.ueg()
                    r.align()
                    r.skip(n)
            r.align()
            pics.append((t, size, fnum, r.bits(QP_BITS), prev_type == PT_META))
        else:
            other += size
        prev_type = t
        at += size
        if t == PT_EOS:
            break
    assert at == len(b)
    return pics, other


def decode(lib, stream, w, h, sub, n):
    bd = L.BatchDecoder(lib, 1)
    try:
        outs, fr = bd.decode([stream], L.frame_bytes(w, h, sub), n)
    finally:
        bd.close()
    assert fr == [n]
    return outs[0]


def plane_sse(a, b, w, h, sub):
    """[sum (a - b)^2] per plane of two packed frames"""
    out, off = [], 0
    for pw, ph in L.plane_dims(w, h, sub):
        x = a[off:off + pw * ph].astype(np.int64)
        y = b[off:off + pw * ph].astype(np.int64)
        out.append(int(((x - y) ** 2).sum()))
        off += pw * ph
    return out


def check(lib, recs, yuv, stream, w, h, fmt, n, inter=True):
    """every record against the stream's packets and numpy's squared error over (input, decoded stream)"""
    sub = L.SUBSAMP[fmt]
    fb = L.frame_bytes(w, h, sub)
    assert recs is not None and len(recs) == n
    pics, other = walk(stream)
    assert len(pics) == n
    assert int(recs["bytes"].sum()) + other == len(stream)
    dec = decode(lib, stream, w, h, sub, n)
    samples = [pw * ph for pw, ph in L.plane_dims(w, h, sub)]
    for r, (t, size, fnum, quant, after_meta) in zip(recs, pics):
        assert (int(r["fnum"]), int(r["is_p"]), int(r["quant"]), int(r["bytes"])) == (fnum, t & 1, quant, size)
        assert int(r["forced_intra"]) == int(inter and not (t & 1) and not after_meta)
        assert list(r["samples"]) == samples
        f = int(r["fnum"])
        want = plane_sse(yuv[f * fb:(f + 1) * fb], dec[f * fb:(f + 1) * fb], w, h, sub)
        assert [int(v) for v in r["sse"]] == want, (f, list(r["sse"]), want)
    return pics
