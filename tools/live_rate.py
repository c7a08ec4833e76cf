"""Rate and latency of live streams (dsvb_enc_push / dsvb_dec_push) against the two other ways to code N feeds.

N feeds of 1920x1080 4:2:0 gop12 (CRF, qp85), T pictures each, made on the GPU by dsvb_synth_device (one seed per
feed) and kept in device memory.  Three arms per direction, one after the other in one process, each after a warm-up:

  encode  live     one DSVB_ENC with N lanes; feed i opens at push (i * gop) // N so that the feeds' I pictures fall on
                   different pushes; every push codes the next picture of every open feed (device pictures in, packets
                   out to pinned host buffers).  Latency = wall time of one dsvb_enc_push call.
          batch    dsvb_encode of the same N x T device pictures in one call (whole sequences, lanes in lock step).
          threads  N DSV_ENCODER objects (dsv_enc through tools/api_harness.c), one per host thread, host pictures
                   (copied from the device once, before timing).  Only the mean time per picture is known.
  decode  live     one DSVB_DEC with N lanes; every push hands each feed's next packet (from the live streams, host
                   memory) and decodes its pictures to device memory.  Latency = wall time of one push that decodes
                   pictures (metadata-only pushes are not counted).
          batch    dsvb_decode of the N streams to device memory in one call.
          threads  N DSV_DECODER objects (dsv_dec), one per host thread, host pictures out.

Pictures/s = N * T over the wall time of the arm.  Prints the card's name and power limit (nvidia-smi, a read) beside
the results, and writes them as JSON to --out.
usage: python tools/live_rate.py [--feeds 16] [--frames 48] [--out live_rate.json]
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import dsvlibs as L  # noqa: E402
import livelibs as LV  # noqa: E402

W, H, FMT, GOP, QP = 1920, 1080, "420", 12, 85


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                           check=True).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in q.split(",")]
        return {"name": name, "power_limit": power}
    except Exception as e:  # the numbers still stand, but say that the card could not be read
        return {"name": "unknown (%s)" % e, "power_limit": "unknown"}


def lat(ms):
    return {"median_ms": statistics.median(ms), "p99_ms": float(np.percentile(ms, 99)), "pushes": len(ms)} if ms else None


def live_encode(gpu, cfg, n, t, d_pics, fb, outs, bound):
    """one pass of the live arm: returns (streams, seconds, per-push ms)"""
    enc = LV.LiveEncoder(gpu, cfg, n)
    streams = [bytearray() for _ in range(n)]
    sid, done = [None] * n, [0] * n
    ms, push = [], 0
    t0 = time.perf_counter()
    while any(d < t for d in done):
        for i in range(n):
            if sid[i] is None and done[i] == 0 and push >= (i * GOP) // n:
                sid[i] = enc.open()
        take = [i for i in range(n) if sid[i] is not None]
        a = time.perf_counter()
        rc, lens = enc.push_ptrs([sid[i] for i in take], [d_pics[i] + done[i] * fb for i in take], 1,
                                 [outs[i].data_ptr() for i in take], [bound] * len(take))
        ms.append((time.perf_counter() - a) * 1e3)
        assert rc == 0, rc
        for k, i in enumerate(take):
            streams[i] += outs[i][:lens[k]].numpy().tobytes()
            done[i] += 1
            if done[i] == t:
                rc, eos = enc.end(sid[i])
                assert rc == 0
                streams[i] += eos
                sid[i] = None
        push += 1
    sec = time.perf_counter() - t0
    enc.close()
    return [bytes(s) for s in streams], sec, ms


def live_decode(gpu, streams, t, d_out, fb):
    """one pass of the live arm: every push hands each feed its next packet; returns (seconds, per-push ms)"""
    n = len(streams)
    dec = LV.LiveDecoder(gpu, n)
    pk = [LV.split_packets(s) for s in streams]
    bufs = [[np.frombuffer(p, dtype=np.uint8) for p in q] for q in pk]
    sid = [dec.open() for _ in range(n)]
    pos, npic, ms = [0] * n, [0] * n, []
    t0 = time.perf_counter()
    while any(p < len(q) for p, q in zip(pos, pk)):
        take = [i for i in range(n) if pos[i] < len(pk[i])]
        pics = sum(1 for i in take if pk[i][pos[i]][5] & 4)
        a = time.perf_counter()
        rc, codes, fnums = dec.push_ptrs([sid[i] for i in take], [bufs[i][pos[i]].ctypes.data for i in take], None,
                                         [len(bufs[i][pos[i]]) for i in take], [d_out[i] + npic[i] * fb for i in take], 1)
        if pics:
            ms.append((time.perf_counter() - a) * 1e3)
        assert rc == 0, rc
        for k, i in enumerate(take):
            npic[i] += codes[k] == LV.DEC_OK and fnums[k] >= 0
            pos[i] += 1
            if pos[i] == len(pk[i]):
                dec.end(sid[i])
    sec = time.perf_counter() - t0
    dec.close()
    assert npic == [t] * n, npic
    return sec, ms


def threaded(fn, n):
    """fn(i) on n threads at once (ctypes releases the GIL inside the library); returns the wall time"""
    th = [threading.Thread(target=fn, args=(i,)) for i in range(n)]
    t0 = time.perf_counter()
    for x in th:
        x.start()
    for x in th:
        x.join()
    return time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--feeds", type=int, default=16)
    ap.add_argument("--frames", type=int, default=48)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    n, t = a.feeds, a.frames
    gpu = L.gpu()
    sub = L.SUBSAMP[FMT]
    fb = L.frame_bytes(W, H, sub)
    cfg = L.make_cfg(W, H, FMT, gop=GOP, qp=QP)
    info = card()
    print("card: %s, power limit %s; %d feeds x %d pictures, %dx%d 4:2:0 gop%d qp%d" % (info["name"], info["power_limit"], n, t, W, H,
                                                                                       GOP, QP), flush=True)
    d_yuv = torch.empty(n * t * fb, dtype=torch.uint8, device="cuda")
    for i in range(n):
        assert gpu.lib.dsvb_synth_device(W, H, sub, 0, t, 500 + i, 0, C.c_void_p(d_yuv.data_ptr() + i * t * fb), 0) == 0
    d_pics = [d_yuv.data_ptr() + i * t * fb for i in range(n)]
    res = {"card": info, "feeds": n, "frames": t, "format": "%dx%d 4:2:0 gop%d qp%d" % (W, H, GOP, QP)}

    # ---- encode ----
    probe = LV.LiveEncoder(gpu, cfg, 1)
    bound = probe.bound
    probe.close()
    outs = [torch.empty(bound, dtype=torch.uint8).pin_memory() for _ in range(n)]
    live_encode(gpu, cfg, min(n, 2), 3, d_pics, fb, outs, bound)                     # warm-up
    streams, sec, ms = live_encode(gpu, cfg, n, t, d_pics, fb, outs, bound)
    res["encode_live"] = {"pictures_per_s": n * t / sec, "latency": lat(ms), "seconds": sec}

    cap = 16 << 20
    sbuf = torch.empty(n * cap, dtype=torch.uint8).pin_memory()
    be = L.BatchEncoder(gpu, cfg, n)
    be.encode_ptrs(d_pics[:1], 2, 1, [sbuf.data_ptr()], [cap])                         # warm-up
    t0 = time.perf_counter()
    rc, lens = be.encode_ptrs(d_pics, t, 1, [sbuf.data_ptr() + i * cap for i in range(n)], [cap] * n)
    sec = time.perf_counter() - t0
    be.close()
    assert rc == 0
    same = all(sbuf[i * cap:i * cap + lens[i]].numpy().tobytes() == streams[i] for i in range(n))
    res["encode_batch"] = {"pictures_per_s": n * t / sec, "latency": "not measured (one call per %d pictures: %.1f ms)" % (n * t, sec * 1e3),
                           "seconds": sec, "streams_equal_live": same}

    host = d_yuv.cpu().numpy()
    seqs = [host[i * t * fb:(i + 1) * t * fb] for i in range(n)]
    gpu.encode_sequence(cfg, seqs[0][:2 * fb], 2)                                        # warm-up
    per = [None] * n

    def enc_one(i):
        per[i] = gpu.encode_sequence(cfg, seqs[i], t)
    sec = threaded(enc_one, n)
    res["encode_threads"] = {"pictures_per_s": n * t / sec, "seconds": sec,
                             "latency": "not measured (mean %.2f ms per picture per feed)" % (1e3 * statistics.mean(p[2] for p in per) / t),
                             "streams_equal_live": all(per[i][0] == streams[i] for i in range(n))}
    del host, seqs, per

    # ---- decode ----
    d_out = torch.empty(n * t * fb, dtype=torch.uint8, device="cuda")
    d_outs = [d_out.data_ptr() + i * t * fb for i in range(n)]
    live_decode(gpu, [streams[0]] * min(n, 2), t, d_outs, fb)                           # warm-up
    sec, ms = live_decode(gpu, streams, t, d_outs, fb)
    res["decode_live"] = {"pictures_per_s": n * t / sec, "latency": lat(ms), "seconds": sec}
    live_pics = d_out.cpu()

    bd = L.BatchDecoder(gpu, n)
    sb = [np.frombuffer(s, dtype=np.uint8) for s in streams]
    bd.decode_ptrs([sb[0].ctypes.data], None, [len(sb[0])], [d_outs[0]], [t * fb], 1)  # warm-up
    t0 = time.perf_counter()
    rc, fr = bd.decode_ptrs([b.ctypes.data for b in sb], None, [len(b) for b in sb], d_outs, [t * fb] * n, 1)
    sec = time.perf_counter() - t0
    bd.close()
    assert rc == 0 and fr == [t] * n
    res["decode_batch"] = {"pictures_per_s": n * t / sec, "seconds": sec, "pictures_equal_live": bool(torch.equal(d_out.cpu(), live_pics)),
                           "latency": "not measured (one call per %d pictures: %.1f ms)" % (n * t, sec * 1e3)}

    gpu.decode_stream(streams[0], W, H, sub, t)                                           # warm-up
    dper = [None] * n

    def dec_one(i):
        nf, pics, _, s = gpu.decode_stream(streams[i], W, H, sub, t)
        dper[i] = (nf == t and np.array_equal(pics, live_pics[i * t * fb:(i + 1) * t * fb].numpy()), s)
    sec = threaded(dec_one, n)
    res["decode_threads"] = {"pictures_per_s": n * t / sec, "seconds": sec, "pictures_equal_live": all(p[0] for p in dper),
                             "latency": "not measured (mean %.2f ms per picture per feed)" % (1e3 * statistics.mean(p[1] for p in dper) / t)}

    for k in ("encode_live", "encode_batch", "encode_threads", "decode_live", "decode_batch", "decode_threads"):
        r = res[k]
        lt = r["latency"]
        lt = "push latency median %.2f ms, p99 %.2f ms over %d pushes" % (lt["median_ms"], lt["p99_ms"], lt["pushes"]) if isinstance(lt, dict) else lt
        print("%-15s %8.0f pictures/s  %s" % (k, r["pictures_per_s"], lt), flush=True)
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
