"""Cost of the encoders' per-picture report (dsvb_enc_set_picture_info) or, with --report ssim, of the SSIM report
(dsvb_enc_set_picture_ssim) on the bench workload.

Configs (bench.py / BASELINE.json): 5 = 1920x1080 4:2:0 gop12, 64 lanes x 12 pictures, device-resident input made by
dsvb_synth_device; 2 = the same with gop 0, where the report adds the whole inverse transform (intra-only pictures are
not references and are otherwise never reconstructed).

  1. Encode calls with the report off and on, alternating, `--reps` times each after one warm-up call of each, in one
     process; host clock around the calls (dsvb_encode returns when the streams are on the host).
  2. A separate pass with live kernel timing: the report kernel's (sse_kernel / ssim_kernel) device time per launch,
     against the time a copy of the same bytes (2 per sample: source and reconstruction) takes at the device-to-device
     copy rate measured here.

Prints the card's name and power limit (nvidia-smi, a read) and writes everything as JSON to --out.
usage: python tools/picture_info_cost.py [--report sse|ssim] [--reps 6] [--out profiles/picture_info_cost.json]
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import picinfo as PI  # noqa: E402  (the report's Python bindings, next to dsvlibs)
import picssim as PS  # noqa: E402  (the SSIM report's)

W, H, FMT, NFR, B = 1920, 1080, "420", 12, 64
# report -> (switch, kernel)
REPORTS = {"sse": (PI.set_picture_info, "sse_kernel"), "ssim": (PS.set_picture_ssim, "ssim_kernel")}


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                           check=True).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in q.split(",")]
        return {"name": name, "power_limit": power}
    except Exception as e:  # the numbers still stand, but say that the card could not be read
        return {"name": "unknown (%s)" % e, "power_limit": "unknown"}


def copy_peak_gbs(torch):
    """device-to-device copy rate of a 1 GiB buffer (read + write bytes over time), best of 10"""
    a = torch.empty(1 << 30, dtype=torch.uint8, device="cuda")
    b = torch.empty_like(a)
    best = 0.0
    for _ in range(12):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        b.copy_(a)
        e1.record()
        e1.synchronize()
        best = max(best, 2 * a.numel() / (e0.elapsed_time(e1) * 1e-3) / 1e9)
    del a, b
    return best


def run_config(L, torch, gpu, gop, reps, peak, report="sse"):
    switch, kname = REPORTS[report]
    sub = L.SUBSAMP[FMT]
    fb = L.frame_bytes(W, H, sub)
    seq = fb * NFR
    d_yuv = torch.empty(B * seq, dtype=torch.uint8, device="cuda")
    for s in range(B):
        gpu.lib.dsvb_synth_device(W, H, sub, 0, NFR, 100 + s, 0, C.c_void_p(d_yuv.data_ptr() + s * seq), 0)
    cap = max(8 << 20, (seq // 3 + 4095) & ~4095)
    h_streams = torch.zeros(B * cap, dtype=torch.uint8).pin_memory()
    enc = L.BatchEncoder(gpu, L.make_cfg(W, H, FMT, gop=gop, qp=85), B)
    yp = [d_yuv.data_ptr() + s * seq for s in range(B)]
    sp = [h_streams.data_ptr() + s * cap for s in range(B)]

    def call(on):
        switch(enc, on)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        rc, lens = enc.encode_ptrs(yp, NFR, 1, sp, [cap] * B)
        dt = time.perf_counter() - t0
        assert rc == 0
        return dt * 1e3, lens

    _, lens_off = call(False)
    _, lens_on = call(True)
    assert lens_off == lens_on
    ms = {False: [], True: []}
    for r in range(reps):
        for on in ((False, True) if r % 2 == 0 else (True, False)):
            ms[on].append(call(on)[0])
    # kernel time, in a pass of its own (timing events slow the steps)
    switch(enc, True)
    enc.set_kernel_timing(True)
    enc.kernel_times(reset=True)
    enc.encode_ptrs(yp, NFR, 1, sp, [cap] * B)
    kt = enc.kernel_times(reset=True)
    recs = PI.picture_info(enc, 0) if report == "sse" else PS.picture_ssim(enc, 0)
    enc.set_kernel_timing(False)
    enc.close()
    kt_rep = kt.get(kname, {"ms": 0.0, "launches": 0})
    k_ms = kt_rep["ms"] / max(kt_rep["launches"], 1)
    step_bytes = 2 * fb * B  # source + reconstruction, every sample of a step's pictures
    off, on = statistics.median(ms[False]), statistics.median(ms[True])
    if report == "sse":
        example = {"example_psnr_y_first_picture": float(PI.psnr(recs["sse"][0][0], recs["samples"][0][0]))}
    else:
        example = {"example_ssim_first_picture": [float(v) for v in recs["ssim"][0]]}
    return {
        "config": "%dx%d %s gop%d, %d lanes x %d pictures, device-resident input" % (W, H, FMT, gop, B, NFR),
        "call_ms_off": ms[False], "call_ms_on": ms[True],
        "median_call_ms_off": off, "median_call_ms_on": on,
        "median_step_ms_off": off / NFR, "median_step_ms_on": on / NFR,
        "delta_pct": 100.0 * (on - off) / off,
        kname + "_ms_per_launch": k_ms, kname + "_launches": kt_rep["launches"],
        report + "_bytes_per_launch": step_bytes,
        report + "_share_of_copy_peak": (step_bytes / (peak * 1e9) * 1e3) / k_ms if k_ms > 0 else None,
        "sbt_inv_kernel_ms": {k: v for k, v in kt.items() if k.startswith("sbt_inv")},
        **example,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--report", choices=sorted(REPORTS), default="sse")
    ap.add_argument("--reps", type=int, default=6)
    ap.add_argument("--out", default=os.path.join("profiles", "picture_info_cost.json"))
    args = ap.parse_args()
    import torch
    import dsvlibs as L
    if not torch.cuda.is_available():
        raise SystemExit("picture_info_cost.py: no CUDA device")
    gpu = L.gpu()
    info = card()
    print("card: %s, power limit %s" % (info["name"], info["power_limit"]))
    peak = copy_peak_gbs(torch)
    kname = REPORTS[args.report][1]
    res = {"card": info, "copy_peak_GBps": peak, "reps": args.reps, "report": args.report, "configs": {}}
    for name, gop in (("5", 12), ("2", 0)):
        r = run_config(L, torch, gpu, gop, args.reps, peak, args.report)
        res["configs"][name] = r
        print("config %s: step %.3f -> %.3f ms (%+.2f %%), %s %.4f ms/launch (%.0f %% of the copy rate %.0f GB/s)" %
              (name, r["median_step_ms_off"], r["median_step_ms_on"], r["delta_pct"], kname, r[kname + "_ms_per_launch"],
               100 * (r[args.report + "_share_of_copy_peak"] or 0), peak))
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
