"""Live streams (dsvb_enc_open / _push / _close, dsvb_dec_open / _push / _close, csrc/host/live.cpp) on the B200: the
golden vectors of the unmodified reference (tests/golden/streams.json) coded as several concurrent copies in one
object, opened at different times and pushed in random subsets, then decoded packet by packet with the copies
interleaved; streams that outnumber the lanes; ABR and intra-only objects; device and host pictures in and out; the
reports; every error path."""
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest

import dsvlibs as L
import livelibs as LV

pytestmark = pytest.mark.gpu

GOLD = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "streams.json")))


@pytest.mark.parametrize("name,copies,stagger", [("cif_gop12", 2, 7), ("qcif_gop12_444", 3, 4), ("qcif_gop12_422", 3, 5),
                                                 ("qcif_gop12_411", 3, 3), ("w854_gop6", 3, 2), ("hd_gop12_qp50", 2, 3)])
def test_live_golden(gpu, name, copies, stagger):
    g = GOLD[name]
    w, h, fmt, n = g["w"], g["h"], g["fmt"], g["frames"]
    sub = L.SUBSAMP[fmt]
    fb = L.frame_bytes(w, h, sub)
    yuv = L.synth_sequence(w, h, fmt, n, g["seed"], g["cut"])
    assert hashlib.md5(yuv.tobytes()).hexdigest() == g["yuv_md5"]
    enc = LV.LiveEncoder(gpu, L.make_cfg(w, h, fmt, gop=g["gop"], qp=g["qp"]), copies)
    try:
        got, where = LV.live_encode(enc, [yuv] * copies, [n] * copies, np.random.default_rng(len(name)), stagger=stagger)
    finally:
        enc.close()
    for s in got:
        assert len(s) == g["dsv_len"] and hashlib.md5(s).hexdigest() == g["dsv_md5"]
    # the copies shared pushes at different pictures of their sequences
    at = [{p: t for t, (p, _) in enumerate(wh)} for wh in where]
    assert any(p in at[1] and at[1][p] != t for p, t in at[0].items())
    dec = LV.LiveDecoder(gpu, copies)
    try:
        pics = LV.live_decode(dec, got, fb, [n] * copies, np.random.default_rng(len(name) + 1))
    finally:
        dec.close()
    for p in pics:
        assert hashlib.md5(p.tobytes()).hexdigest() == g["dec_md5"]


def test_live_lanes_reused_mixed_phases(gpu):
    """seven streams of different seeds, lengths and scene cuts through three lanes"""
    specs = [(20, 101, 0), (9, 102, 4), (30, 103, 13), (5, 104, 0), (14, 105, 0), (26, 106, 20), (12, 107, 1)]
    LV.check_mixed_streams(gpu, 352, 288, "420", 3, specs, 1, gop=12)
    LV.check_mixed_streams(gpu, 640, 360, "422", 2, specs[:4], 2, gop=6, qp=70)


def test_live_abr(gpu):
    """ABR: every stream's quantisers follow its own packet sizes"""
    specs = [(24, 111, 9), (16, 112, 0), (20, 113, 0), (10, 114, 3)]
    LV.check_mixed_streams(gpu, 352, 288, "420", 3, specs, 3, gop=12, rc_mode=1, bitrate=800000,
                           quality=L.qp_to_quality(70) * 3 // 2)


def test_live_intra_only(gpu):
    specs = [(6, 121, 0), (4, 122, 0), (7, 123, 2)]
    LV.check_mixed_streams(gpu, 640, 360, "420", 2, specs, 4, gop=0)


def test_live_device_and_host_io(gpu):
    """device pictures in (torch tensors); pinned host pictures in and a pinned output; decode with device packet copies
    to device pictures and without them to host pictures, against dsvb_decode"""
    import torch
    w, h, fmt, n = 640, 360, "420", 14
    sub = L.SUBSAMP[fmt]
    fb = L.frame_bytes(w, h, sub)
    cfg = L.make_cfg(w, h, fmt, gop=12)
    seeds = [(131, 0), (132, 5), (133, 0)]
    d_yuv = []
    for s, c in seeds:
        d = torch.zeros(fb * n, dtype=torch.uint8, device="cuda")
        assert gpu.lib.dsvb_synth_device(w, h, sub, 0, n, s, c, C.c_void_p(d.data_ptr()), 0) == 0
        d_yuv.append(d)
    host = [L.synth_sequence(w, h, fmt, n, s, c) for s, c in seeds]
    want = [gpu.encode_sequence(cfg, q, n)[0] for q in host]
    enc = LV.LiveEncoder(gpu, cfg, 3)
    try:
        got, _ = LV.live_encode(enc, None, [n] * 3, np.random.default_rng(5), stagger=4, on_device=True,
                                pics=lambda i, t: d_yuv[i].data_ptr() + t * fb)
        assert got == want
        hp = torch.from_numpy(host[1]).pin_memory()
        out = torch.zeros(enc.bound, dtype=torch.uint8).pin_memory()
        sid, s = enc.open(), b""
        for t in range(n):
            rc, lens = enc.push_ptrs([sid], [hp.data_ptr() + t * fb], 0, [out.data_ptr()], [enc.bound])
            assert rc == 0
            s += out[:lens[0]].numpy().tobytes()
        rc, eos = enc.end(sid)
        assert rc == 0 and s + eos == want[1]
    finally:
        enc.close()
    bd = L.BatchDecoder(gpu, 3)
    ref, fr = bd.decode(want, fb, n)
    bd.close()
    assert fr == [n] * 3
    pk = [LV.split_packets(s) for s in want]
    d_pk = [[torch.from_numpy(np.frombuffer(p, dtype=np.uint8).copy()).cuda() for p in q] for q in pk]
    d_out = [torch.zeros(fb * n, dtype=torch.uint8, device="cuda") for _ in want]
    h_out = np.zeros(fb * n, dtype=np.uint8)
    dec = LV.LiveDecoder(gpu, 3)
    try:
        sid = [dec.open() for _ in want]
        npic = [0, 0, 0]
        for j in range(max(len(q) for q in pk)):
            for group, on_dev in (([0, 1], 1), ([2], 0)):
                take = [i for i in group if j < len(pk[i])]
                if not take:
                    continue
                bufs = [np.frombuffer(pk[i][j], dtype=np.uint8) for i in take]
                outs = [(d_out[i].data_ptr() if on_dev else h_out.ctypes.data) + npic[i] * fb for i in take]
                devs = [d_pk[i][j].data_ptr() for i in take] if on_dev else None
                rc, codes, fnums = dec.push_ptrs([sid[i] for i in take], [b.ctypes.data for b in bufs], devs,
                                                 [len(b) for b in bufs], outs, on_dev)
                assert rc == 0
                for k, i in enumerate(take):
                    if codes[k] == LV.DEC_OK:
                        assert fnums[k] == npic[i]
                        npic[i] += 1
        assert npic == [n] * 3
        st = dec.stats()
    finally:
        dec.close()
    torch.cuda.synchronize()
    for i in (0, 1):
        assert np.array_equal(d_out[i].cpu().numpy(), ref[i])
    assert np.array_equal(h_out, ref[2])
    assert st["h2d_bytes"] == sum(len(p) for p in pk[2] if p[5] & 4)   # only stream 2's picture packets crossed PCIe


@pytest.mark.parametrize("draw,to420", [(7, 1), (7, 0), (0, 1)])
def test_live_decoder_output_options(gpu, draw, to420):
    """dsvb_dec_set_draw_info / _set_out420p on live decoding equal dsvb_decode with the same settings"""
    g = GOLD["qcif_gop12_444"]
    w, h, fmt, n = g["w"], g["h"], g["fmt"], g["frames"]
    sub = L.SUBSAMP[fmt]
    stream = gpu.encode_sequence(L.make_cfg(w, h, fmt, gop=g["gop"], qp=g["qp"]),
                                 L.synth_sequence(w, h, fmt, n, g["seed"], g["cut"]), n)[0]
    fbo = L.frame_bytes(w, h, L.SUBSAMP["420"] if to420 else sub)
    bd = L.BatchDecoder(gpu, 2)
    bd.set_draw_info(draw)
    bd.set_out420p(to420)
    want, fr = bd.decode([stream], fbo, n)
    bd.close()
    assert fr == [n]
    dec = LV.LiveDecoder(gpu, 2)
    dec.set_draw_info(draw)
    dec.set_out420p(to420)
    try:
        pics = LV.live_decode(dec, [stream, stream], fbo, [n, n], np.random.default_rng(draw + to420))
    finally:
        dec.close()
    assert np.array_equal(pics[0], want[0]) and np.array_equal(pics[1], want[0])


def test_live_reports(gpu):
    LV.check_reports(gpu, 352, 288, "420", 14, 3, 140, gop=12)
    LV.check_reports(gpu, 176, 144, "444", 5, 2, 150, gop=0)


def test_live_encoder_errors(gpu):
    LV.check_encoder_errors(gpu, 176, 144, "420")


def test_live_decoder_errors(gpu):
    LV.check_decoder_errors(gpu, 176, 144, "420", 352, 288)
