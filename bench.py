#!/usr/bin/env python3
"""bench.py -- DSV1 encode+decode throughput on B200 (BASELINE.json metric), one process per GPU.

Workload (config.workload): per GPU a batch of B synthetic 1920x1080 4:2:0 closed-GOP sequences (12 pictures,
-gop12 -qp85 fixed quality, hierarchical ME with auto pyramid depth) -- BASELINE.json config 5 sharded by
sequence, weak scaling: every rank encodes AND decodes its own B sequences, no collective on the data path.
A "step" = encode all B*12 pictures to .dsv streams, then decode those streams back to pictures.

  value   pictures/s through encode+decode with the inputs of each direction already resident in HBM
          (pictures generated on the device; streams also kept on the device for the decoder; decoded
          pictures left on the device).  Bitstreams still come back to the host: that IS the encoder's product.
  e2e     the same through the same public call with HOST buffers (pinned): pictures H2D, streams D2H,
          streams H2D, pictures D2H all inside the timed region.
  roofline  the kernel with the largest total time in the device-resident timed region; `kernels` lists every
          kernel >= 1 % of the step.  Every launch is bracketed by CUDA events on the engine's stream
          (csrc/ktime.cu): algorithmic bytes / duration.  `traffic` comes from profiles/traffic.json (parsed
          from a committed ncu --set full capture) or is null.
  encode_/decode_pictures_per_s  the two directions of the device-resident step separately (N=1).
  verified  the cpu_baseline leg's reference streams / pictures are compared with the GPU's for the same
          sequences; on a mismatch no line is printed.
  --config 2|3|4|5  BASELINE.json configs (5 = headline metric, default).
  cpu_baseline  the UNMODIFIED reference (oracle/_ref/libdsv1ref.so, built by oracle/Makefile from the reference's
          source tree, its REF) single-threaded on a bounded sample of the same workload, rank 0, N=1.

`--dump-outputs DIR` writes, after the timed steps, what the last device-resident step returned to its caller (rank 0's
sequences): stream_lengths.npy (float64, one per sequence), streams_sample.npy (float32, sequences x a fixed, seeded set
of relative positions in each stream) and pictures_sample.npy (float32, sequences x pictures x a fixed, seeded set of
byte positions in the decoded picture), together at most 64 MB.  The inputs depend on the arguments only, so two builds
run with the same arguments can be compared output for output.  Two limits: the timed decoder decodes the streams of
the untimed first step (parked in HBM before timing), so pictures_sample.npy reflects the encoder of that step and the
timed encoder shows only in the streams; and the stream positions are fractions of each stream's own length, so a
stream whose length changed is caught by stream_lengths.npy but its sampled bytes no longer line up byte for byte.

`--impl reference` times the reference's own CPU implementation on all host cores (one process per core, the
reference is not thread-safe), same metric / unit / config.
"""
import argparse
import ctypes as C
import json
import multiprocessing as mp
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "tests"))

W, H, FMT, GOP, QP, NFR = 1920, 1080, "420", 12, 85, 12
METRIC = "1080p 4:2:0 gop12 qp85 encode+decode pictures/s (bit-exact DSV1)"
# BASELINE.json configs[1..4] (index = --config).  5 is the headline (the metric is quoted on it); 2-4 are the
# reference's single-sequence operating points (dsv_main.c:463-489) run as a batch of independent sequences.
CONFIGS = {
    2: dict(w=1920, h=1080, fmt="420", gop=0, nfr=12, batch=64, tag="BASELINE config 2, -gop0 intra-only",
            metric="1080p 4:2:0 gop0 (intra-only) qp85 encode+decode pictures/s (bit-exact DSV1)"),
    3: dict(w=1920, h=1080, fmt="420", gop=12, nfr=24, batch=32, tag="BASELINE config 3, -gop12 inter, 24-picture sequences",
            metric="1080p 4:2:0 gop12 qp85 encode+decode pictures/s, 24-picture sequences (bit-exact DSV1)"),
    4: dict(w=3840, h=2160, fmt="444", gop=12, nfr=6, batch=16, tag="BASELINE config 4, 2160p 4:4:4 -gop12",
            metric="2160p 4:4:4 gop12 qp85 encode+decode pictures/s (bit-exact DSV1)"),
    5: dict(w=1920, h=1080, fmt="420", gop=12, nfr=12, batch=64, tag="BASELINE config 5, sharded by sequence",
            metric=METRIC),
}


def select_config(args):
    global W, H, FMT, GOP, NFR, METRIC
    c = CONFIGS[args.config]
    W, H, FMT, GOP, NFR, METRIC = c["w"], c["h"], c["fmt"], c["gop"], c["nfr"], c["metric"]
    if args.batch is None:
        args.batch = c["batch"]
    args.tag = c["tag"]


def workload(batch, tag="BASELINE config 5, sharded by sequence"):
    import dsvlibs as L
    fb = L.frame_bytes(W, H, L.SUBSAMP[FMT])
    return {"workload": "synthetic %dx%d %s, %d closed-GOP sequences x %d pictures per GPU, -gop%d -qp%d CRF, "
                        "encode then decode (%s)" % (W, H, FMT, batch, NFR, GOP, QP, tag),
            "batch_sequences_per_gpu": batch, "pictures_per_sequence": NFR,
            "l2": "inputs larger than L2 (%.0f MB of pictures per step per GPU)" % (batch * NFR * fb / 1e6)}


# ------------------------------------------------------------------------------------------------------
# reference arm / cpu baseline
# ------------------------------------------------------------------------------------------------------
_REF_STATE = {}


def _ref_init(seed_base):
    """per-process: load the reference library and synthesise this process's input sequence once (untimed)"""
    import dsvlibs as L
    ident = mp.current_process()._identity
    seed = seed_base + (ident[0] if ident else 0)
    _REF_STATE["ref"] = L.ref()
    _REF_STATE["yuv"] = L.synth_sequence(W, H, FMT, NFR, seed, 0)
    _REF_STATE["cfg"] = L.make_cfg(W, H, FMT, gop=GOP, qp=QP)


def _ref_codec(yuv, keep=False):
    import dsvlibs as L
    ref = _REF_STATE.get("ref") or L.ref()
    cfg = _REF_STATE.get("cfg") or L.make_cfg(W, H, FMT, gop=GOP, qp=QP)
    stream, _, e = ref.encode_sequence(cfg, yuv, NFR)
    nf, dec, _, d = ref.decode_stream(stream, W, H, L.SUBSAMP[FMT], NFR)
    assert nf == NFR
    return (e, d, stream, dec) if keep else (e, d)


def _ref_step(_):
    return _ref_codec(_REF_STATE["yuv"])


def run_reference(args):
    import dsvlibs as L
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if not L.have_ref():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libdsv1ref.so missing (built by oracle/Makefile from the reference's source tree)"}))
        return
    cores = os.cpu_count() or 1
    procs = max(1, min(cores, 64))
    pool = mp.get_context("fork").Pool(procs, initializer=_ref_init, initargs=(1000,))
    pool.map(_ref_step, range(procs))  # every worker is up and has its input
    times = []
    nseq = args.batch  # the product arm's step: `batch` sequences, spread over the host cores
    pics = nseq * NFR
    for it in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        pool.map(_ref_step, range(nseq), chunksize=1)
        dt = time.perf_counter() - t0
        if it >= args.warmup:
            times.append(dt)
    pool.close()
    total = sum(times)
    value = pics * len(times) / total
    line = {"metric": METRIC, "value": value, "unit": "pictures/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8/int32", "data": "synthetic", "impl": "reference",
            "config": workload(args.batch, args.tag),
            "cpu_baseline": {"value": value, "unit": "pictures/s", "cores": procs, "kind": "reference",
                             "sample": "%d sequences x %d pictures per step, encode then decode, spread over %d processes "
                                       "(one per host core; the reference is single-threaded and not re-entrant), each "
                                       "process re-coding its own preloaded sequence" % (nseq, NFR, procs)},
            "e2e": {"value": value, "unit": "pictures/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def cpu_baseline_single(h_yuv_np, seq_bytes):
    """Reference, 1 thread, bounded sample of the SAME inputs: time inside dsv_enc / dsv_dec only."""
    import dsvlibs as L
    if not L.have_ref():
        return None, []
    nseq = min(max(1, int(6 * (1920 * 1080 * 1.5 * 12) / seq_bytes)), 6, len(h_yuv_np) // seq_bytes)
    e = d = 0.0
    kept = []
    for s in range(nseq):
        es, ds, stream, dec = _ref_codec(h_yuv_np[s * seq_bytes:(s + 1) * seq_bytes], keep=True)
        e += es
        d += ds
        kept.append((stream, dec))
    return {"value": nseq * NFR / (e + d), "unit": "pictures/s", "cores": 1, "kind": "reference",
            "encode_pictures_per_s": nseq * NFR / e, "decode_pictures_per_s": nseq * NFR / d,
            "sample": "%d of the step's sequences x %d pictures, 1 thread, time inside dsv_enc+dsv_dec "
                      "(encode %.2f pictures/s, decode %.2f pictures/s)" % (nseq, NFR, nseq * NFR / e, nseq * NFR / d)}, kept


# ------------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows = []
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                       "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.p = None

    def _read(self):
        for line in self.p.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=2)
        except Exception:
            self.p.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nme, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------
# product arm
# ------------------------------------------------------------------------------------------------------
def _cpulist(txt):
    cpus = set()
    for part in txt.strip().split(","):
        if not part:
            continue
        a, _, b = part.partition("-")
        cpus.update(range(int(a), int(b or a) + 1))
    return cpus


def bind_near_gpu(torch, local, world):
    """One process per GPU: run this rank's host threads (and first-touch its pinned staging memory) on the CPUs of
    the NUMA node the GPU hangs off, and size the library's host thread pool to this rank's share of the cores.
    Pure placement -- no effect on results."""
    note = "none"
    try:
        try:
            pr = torch.cuda.get_device_properties(local)
            bdf = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        except AttributeError:
            q = subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                               capture_output=True, text=True, timeout=20).stdout.strip().lower()
            dom, rest = q.split(":", 1)
            bdf = dom[-4:] + ":" + rest
        cpus = _cpulist(open("/sys/bus/pci/devices/%s/local_cpulist" % bdf).read()) & os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            note = "numa-local cpus (%d)" % len(cpus)
    except Exception as e:  # topology not exposed: leave the scheduler alone
        note = "unbound (%s)" % type(e).__name__
    share = max(2, min(8, len(os.sched_getaffinity(0)) * (1 if world == 1 else 2) // max(1, world)))
    os.environ.setdefault("DSV_HOST_THREADS", str(share))
    return note + ", host threads %s" % os.environ["DSV_HOST_THREADS"]



# kernel name -> (bound, algorithmic bytes per PICTURE as f(geometry) or None, which pictures pass through it)
def kernel_models(L):
    sub = L.SUBSAMP[FMT]
    fb = L.frame_bytes(W, H, sub)
    planes, coefs = L.plane_dims(W, H, sub), L.coef_dims(W, H, sub)
    sbt = sum(pw * ph for pw, ph in planes) + 4 * sum(cw * ch for cw, ch in coefs)
    coef4 = 4 * sum(cw * ch for cw, ch in coefs)
    return {
        "sbt_fwd_tile_kernel": ("hbm", sbt), "sbt_inv_tile_kernel": ("hbm", sbt), "sbt_inv_tile_intra_kernel": ("hbm", sbt),
        "bmc_kernel": ("hbm", None), "hzdec_clean_kernel": ("hbm", None),
        # the pack passes read the chunks that hold something (sparse) or the scan pass's lists (dense): no per-picture byte model
        "hzcc_scan_kernel": ("hbm", coef4), "hzcc_pack_kernel": ("latency", None), "hzcc_pack_dense_kernel": ("issue", None),
        "zero_kernel": ("hbm", None),
        "ingest_kernel": ("hbm", 2 * fb), "pack_kernel": ("hbm", 2 * fb), "down2_kernel": ("hbm", None),
        "hme_l0_kernel": ("issue", 2 * fb), "hme_level_kernel": ("issue", None), "hme_neigh_kernel": ("latency", None),
    }


def kernel_table(L, B, steps, ms_dev, peak, es, ds, ekt, dkt):
    """every kernel that takes >= 1 % of the device-resident step: live CUDA-event time (events around each launch on
    the engine's stream), launches, share of the step, and for the streaming kernels algorithmic GB/s vs the measured peak"""
    models = kernel_models(L)
    sub = L.SUBSAMP[FMT]
    fb = L.frame_bytes(W, H, sub)
    sbt = models["sbt_fwd_tile_kernel"][1]
    pictures = B * NFR * steps
    n_i = B * steps * (NFR if GOP == 0 else -(-NFR // GOP))  # no scene cuts in the bench content: I pictures = GOP starts
    n_p = pictures - n_i
    # the inverse transform of P pictures and of I pictures are separate kernels (different occupancy); the encoder's
    # inverse of a P picture also reads the prediction it adds on the way out
    exact = {("enc", "sbt_fwd_tile_kernel"): sbt * pictures,
             ("enc", "sbt_inv_tile_kernel"): (sbt + fb) * n_p, ("dec", "sbt_inv_tile_kernel"): sbt * n_p,
             ("enc", "sbt_inv_tile_intra_kernel"): sbt * n_i, ("dec", "sbt_inv_tile_intra_kernel"): sbt * n_i,
             ("enc", "bmc_kernel"): es["bmc_bytes"], ("dec", "bmc_kernel"): ds["bmc_bytes"]}
    if GOP == 0:  # intra-only: nothing is reconstructed in the encoder
        exact[("enc", "sbt_inv_tile_intra_kernel")] = None
    out = {}
    for side, kt in (("enc", ekt), ("dec", dkt)):
        for name, v in kt.items():
            if v["ms"] < 0.01 * ms_dev:
                continue
            bound, per_pic = models.get(name, ("latency", None))
            by = exact.get((side, name), per_pic * pictures if per_pic else None)
            row = {"ms_total": v["ms"], "launches": v["launches"], "ms_per_launch": v["ms"] / v["launches"],
                   "share_of_step": v["ms"] / ms_dev, "bound": bound}
            if by:
                row.update(bytes_per_launch=by / v["launches"], achieved_gbs=by / v["ms"] / 1e6, frac=by / v["ms"] / 1e6 / peak)
            out["%s(%s)" % (name, side)] = row
    return out


def measured_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch, parsed by tools/ncu_traffic.py from an `ncu --set full`
    capture of this workload and committed as profiles/traffic.json; absent -> no traffic claim"""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        return {}


def dump_outputs(path, np, torch, d_out, h_streams, cap, lens, seq_bytes):
    """a fixed, seeded sample of the streams and decoded pictures of the last step (see --dump-outputs), <= 64 MB"""
    B = len(lens)
    k = max(1, min(65536, (16 << 20) // (4 * B)))
    m = max(1, min(8192, (40 << 20) // (4 * B * NFR)))
    fb = seq_bytes // NFR
    u = np.random.default_rng(0).random(k)
    hs = h_streams.numpy()
    streams = np.stack([hs[s * cap + (u * lens[s]).astype(np.int64)] for s in range(B)]).astype(np.float32)
    pos = np.sort(np.random.default_rng(1).choice(fb, size=min(m, fb), replace=False))
    idx = (torch.arange(B * NFR, device=d_out.device)[:, None] * fb + torch.from_numpy(pos).to(d_out.device)[None, :]).reshape(-1)
    pictures = d_out[idx].cpu().numpy().reshape(B, NFR, len(pos)).astype(np.float32)
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "stream_lengths.npy"), np.asarray(lens, dtype=np.float64))
    np.save(os.path.join(path, "streams_sample.npy"), streams)
    np.save(os.path.join(path, "pictures_sample.npy"), pictures)


def run_product(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    import dsvlibs as L

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product has no CPU path")
    torch.cuda.set_device(local)
    pin_note = bind_near_gpu(torch, local, world)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"  # keep NCCL's version banner off stdout: rank 0 prints ONE JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    gpu = L.gpu()
    lib = gpu.lib
    B = args.batch
    sub = L.SUBSAMP[FMT]
    fb = L.frame_bytes(W, H, sub)
    seq_bytes = fb * NFR
    cfg = L.make_cfg(W, H, FMT, gop=GOP, qp=QP)

    # inputs: generated on the device (SURVEY Appendix C content), one distinct sequence per lane
    d_yuv = torch.empty(B * seq_bytes, dtype=torch.uint8, device="cuda")
    for s in range(B):
        lib.dsvb_synth_device(W, H, sub, 0, NFR, 100 + rank * B + s, 0, C.c_void_p(d_yuv.data_ptr() + s * seq_bytes), local)
    h_yuv = torch.empty(B * seq_bytes, dtype=torch.uint8).pin_memory()
    h_yuv.copy_(d_yuv)
    cap = max(8 << 20, (seq_bytes // 3 + 4095) & ~4095)
    h_streams = torch.zeros(B * cap, dtype=torch.uint8).pin_memory()
    d_streams = torch.zeros(B * cap, dtype=torch.uint8, device="cuda")
    d_out = torch.empty(B * seq_bytes, dtype=torch.uint8, device="cuda")
    h_out = torch.empty(B * seq_bytes, dtype=torch.uint8).pin_memory()

    enc = L.BatchEncoder(gpu, cfg, B, local)
    dec = L.BatchDecoder(gpu, B, local)
    sp = [h_streams.data_ptr() + s * cap for s in range(B)]
    sdp = [d_streams.data_ptr() + s * cap for s in range(B)]
    caps = [cap] * B

    split = {"enc_s": 0.0, "dec_s": 0.0}

    def step(host):
        t0 = time.perf_counter()
        if host:
            rc, lens = enc.encode_ptrs([h_yuv.data_ptr() + s * seq_bytes for s in range(B)], NFR, 0, sp, caps)
            assert rc == 0
            t1 = time.perf_counter()
            rc, fr = dec.decode_ptrs(sp, None, lens, [h_out.data_ptr() + s * seq_bytes for s in range(B)], [seq_bytes] * B, 0)
        else:
            rc, lens = enc.encode_ptrs([d_yuv.data_ptr() + s * seq_bytes for s in range(B)], NFR, 1, sp, caps)
            assert rc == 0
            t1 = time.perf_counter()
            rc, fr = dec.decode_ptrs(sp, sdp, lens, [d_out.data_ptr() + s * seq_bytes for s in range(B)], [seq_bytes] * B, 1)
        assert rc == 0 and all(f == NFR for f in fr), (rc, fr)
        split["enc_s"] += t1 - t0   # both calls return when their products are complete (streams on the host /
        split["dec_s"] += time.perf_counter() - t1   # pictures at their destination)
        return lens

    # end-to-end arm: software-pipelined the way a transcoding service runs.  In every tick one host thread encodes step t
    # while a second one decodes step t-1, both started together and joined before the next tick, so pictures leave the GPU
    # (D2H) while the next ones arrive (H2D) -- PCIe is full duplex, a strictly sequential encode-then-decode uses one
    # direction at a time.  Same public calls, same work, same bytes; every one of the K steps starts and completes inside
    # the timed region (pipeline fill and drain included).  (Free-running encoder / decoder threads coupled only through
    # buffer availability measure the same on the same box: 11.73k / 11.81k against 11.59k / 11.83k pictures/s.)
    # --e2e-parts P > 1 deals the step's sequences to P smaller engine pairs (shorter fill / drain, but smaller launches:
    # measured slower).
    P = max(1, min(args.e2e_parts, B)) if args.e2e_pipeline else 1
    while B % P:
        P -= 1
    n_part = B // P
    if args.e2e_pipeline and P > 1:
        part_enc = [L.BatchEncoder(gpu, cfg, n_part, local) for _ in range(P)]
        part_dec = [L.BatchDecoder(gpu, n_part, local) for _ in range(P)]
    else:
        part_enc, part_dec = [enc], [dec]
    h_streams2 = torch.zeros(B * cap, dtype=torch.uint8).pin_memory() if (args.e2e_pipeline and P == 1) else None
    sp_alt = [h_streams2.data_ptr() + s * cap for s in range(B)] if h_streams2 is not None else None

    def run_pipelined(steps):
        import threading
        lens_all = [None] * B
        errs = []
        ntask = steps * P  # task j = part j % P of step j // P

        def seqs(j):
            p = j % P
            return range(p * n_part, (p + 1) * n_part)

        def stream_ptrs(j):
            # one part per buffer slice; with a single part the two halves of a double buffer alternate
            base = sp if (P > 1 or (j % 2) == 0) else sp_alt
            return [base[s] for s in seqs(j)]

        def do_enc(j):
            try:
                rc, ln = part_enc[j % P].encode_ptrs([h_yuv.data_ptr() + s * seq_bytes for s in seqs(j)], NFR, 0, stream_ptrs(j),
                                                     [cap] * n_part)
                assert rc == 0, rc
                for s, v in zip(seqs(j), ln):
                    lens_all[s] = v
            except BaseException as e:  # noqa: BLE001
                errs.append(e)

        def do_dec(j):
            try:
                rc, fr = part_dec[j % P].decode_ptrs(stream_ptrs(j), None, [lens_all[s] for s in seqs(j)],
                                                     [h_out.data_ptr() + s * seq_bytes for s in seqs(j)], [seq_bytes] * n_part, 0)
                assert rc == 0 and all(f == NFR for f in fr), (rc, fr)
            except BaseException as e:  # noqa: BLE001
                errs.append(e)

        for t in range(ntask + 1):
            th = []
            if t < ntask:
                th.append(threading.Thread(target=do_enc, args=(t,)))
            if t >= 1:
                th.append(threading.Thread(target=do_dec, args=(t - 1,)))
            for x in th:
                x.start()
            for x in th:
                x.join()
            if errs:
                raise errs[0]
        return list(lens_all)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(host, steps, warmup, kernel_timing=False):
        # per-launch timing events are off in the throughput passes (their timestamps cross PCIe, which costs every
        # launch ~40 us next to saturated picture traffic) and on in the pass that builds the kernel table
        enc.set_kernel_timing(kernel_timing)
        dec.set_kernel_timing(kernel_timing)
        for _ in range(warmup):
            lens = run_pipelined(1) if (host and args.e2e_pipeline) else step(host)  # warm the engines the timed region uses
        enc.stats(reset=True)
        dec.stats(reset=True)
        enc.kernel_times(reset=True)
        dec.kernel_times(reset=True)
        split["enc_s"] = split["dec_s"] = 0.0
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        if host and args.e2e_pipeline:
            lens = run_pipelined(steps)
        else:
            for _ in range(steps):
                lens = step(host)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), lens, enc.stats(), dec.stats(), enc.kernel_times(), dec.kernel_times(), dict(split)

    # first pass through the host arm; its (deterministic) streams are then parked in HBM for the decoder's
    # resident-input arm
    lens = step(True)
    d_streams.copy_(h_streams, non_blocking=False)
    torch.cuda.synchronize()
    sampler = ClockSampler(local) if rank == 0 else None
    ms_dev, lens, _, _, _, _, split_dev = timed(False, args.steps, args.warmup)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, np, torch, d_out, h_streams, cap, lens, seq_bytes)
    ms_e2e, lens_h, es_h, ds_h, _, _, _ = timed(True, args.steps, args.warmup)
    # the same device-resident steps once more with every launch bracketed by timing events: kernel table + roofline
    ms_prof, _, es, ds, ekt, dkt, _ = timed(False, args.steps, 1, kernel_timing=True)
    enc.set_kernel_timing(False)
    dec.set_kernel_timing(False)

    # PCIe floor of one end-to-end step on this box: the step's pictures H2D and D2H at the same time, nothing else
    def pcie_floor():
        s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
        best = None
        for _ in range(3):
            barrier()
            t0 = time.perf_counter()
            with torch.cuda.stream(s1):
                d_yuv.copy_(h_yuv, non_blocking=True)
            with torch.cuda.stream(s2):
                h_out.copy_(d_out, non_blocking=True)
            torch.cuda.synchronize()
            dt = (time.perf_counter() - t0) * 1e3
            best = dt if best is None or dt < best else best
        t = torch.tensor([best], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())
    floor_ms = pcie_floor()

    pics = B * NFR * world
    value = pics * args.steps / (ms_dev / 1e3)
    e2e = pics * args.steps / (ms_e2e / 1e3)
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
        kern = kernel_table(L, B, args.steps, ms_prof, peak, es, ds, ekt, dkt)
        dom = max(kern.items(), key=lambda kv: kv[1]["ms_total"]) if kern else (None, None)
        traffic = measured_traffic()
        roofline = None
        if dom[0]:
            k = dom[1]
            tr = traffic.get(dom[0].split("(")[0])
            roofline = {"kernel": dom[0], "bound": "hbm", "limited_by": k["bound"],
                        "achieved": k.get("achieved_gbs"), "peak": peak, "unit": "GB/s", "frac": k.get("frac"),
                        "traffic": (tr["dram_bytes_per_launch"] if tr else None), "traffic_source": (tr["source"] if tr else None),
                        "peak_source": peak_src,
                        "algorithmic_bytes": "per picture: SBT w*h (u8) + 4*cw*ch (int32) per plane (+ w*h prediction read in the encoder's "
                                             "inverse of a P picture); BMC 4 B (encoder) / 3 B (decoder) per sample; HZCC scan and pack "
                                             "4*cw*ch each; HME level 0: source + reference luma and chroma once (2 x frame bytes)",
                        "north_star_kernels": {n: round(v["frac"], 3) for n, v in kern.items()
                                               if v.get("frac") is not None and (n.startswith("sbt_") or n.startswith("bmc_"))}}
        stream_bytes = sum(lens_h)
        line = {"metric": METRIC, "value": value, "unit": "pictures/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "u8/int32", "data": "synthetic",
                "config": workload(B, args.tag),
                "encode_pictures_per_s": pics * args.steps / split_dev["enc_s"] if world == 1 else None,
                "decode_pictures_per_s": pics * args.steps / split_dev["dec_s"] if world == 1 else None,
                "e2e": {"value": e2e, "unit": "pictures/s", "ms_per_step": ms_e2e / args.steps,
                        "h2d_bytes_per_step": B * seq_bytes + stream_bytes, "d2h_bytes_per_step": B * seq_bytes + stream_bytes,
                        "pcie_floor_ms": floor_ms,
                        "pcie_floor_note": "this step's pictures copied H2D and D2H at the same time from / to the same pinned "
                                           "buffers, nothing else running (max over ranks, all ranks copying at once)",
                        "schedule": ("ticks: one host thread encodes step t while a second decodes step t-1 (started together, joined per "
                                     "tick; %d engine pair(s) of %d lanes, double-buffered streams): full-duplex PCIe, pipeline fill and "
                                     "drain inside the timed region" % (P, n_part)) if args.e2e_pipeline
                                    else "encode then decode, one step at a time"},
                "gpu_launches": int(es["kernel_launches"] + ds["kernel_launches"]),
                "roofline": roofline, "kernels": kern,
                "kernels_pass": {"ms_per_step": ms_prof / args.steps,
                                 "note": "the kernel table and the roofline come from a second device-resident pass of the same "
                                         "steps with every launch bracketed by timing events; value / e2e are measured without them"},
                "clocks": clocks, "host_placement": pin_note,
                "stream_bytes_per_step": stream_bytes}
        if world == 1 and not args.no_cpu:
            # the reference codes a sample of the very sequences the timed steps just processed; its streams and
            # decoded pictures must equal the bytes the GPU produced for them in the last timed host-buffer step
            line["cpu_baseline"], kept = cpu_baseline_single(h_yuv.numpy(), seq_bytes)
            last = h_streams2 if (h_streams2 is not None and args.steps % 2 == 0) else h_streams
            hs_np, ho_np = last.numpy(), h_out.numpy()
            for s_i, (r_stream, r_dec) in enumerate(kept):
                g_stream = bytes(hs_np[s_i * cap:s_i * cap + lens_h[s_i]])
                if g_stream != r_stream:
                    raise SystemExit("bench.py: stream of sequence %d differs from the reference (%d vs %d bytes) -- no number printed"
                                     % (s_i, len(g_stream), len(r_stream)))
                if not np.array_equal(ho_np[s_i * seq_bytes:(s_i + 1) * seq_bytes], r_dec):
                    raise SystemExit("bench.py: decoded pictures of sequence %d differ from the reference -- no number printed" % s_i)
            line["verified"] = {"sequences": len(kept), "pictures": len(kept) * NFR,
                                "what": "streams byte-for-byte and decoded pictures sample-for-sample equal to the unmodified reference "
                                        "for the first %d sequences of the last timed host-buffer step" % len(kept)}
        print(json.dumps(line))
    for x in set(part_enc + part_dec + [enc, dec]):
        x.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="product", choices=["product", "reference"])
    ap.add_argument("--batch", type=int, default=None, help="sequences per GPU per step (default: the config's)")
    ap.add_argument("--config", type=int, default=5, choices=sorted(CONFIGS), help="BASELINE.json configs index (5 = headline)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--e2e-parts", type=int, default=1,
                    help="e2e arm: engine pairs the step's sequences are dealt to (measured on one B200, 64 sequences: 1 -> 63 ms per "
                         "step, 2 -> 69, 4 -> 82, 8 -> 109: small engines lose more than the shorter pipeline fill wins)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write a fixed sample of the last device-resident step's streams and decoded pictures to DIR/*.npy")
    ap.add_argument("--no-e2e-pipeline", dest="e2e_pipeline", action="store_false",
                    help="e2e arm: strictly one step at a time instead of decode(k) overlapping encode(k+1)")
    args = ap.parse_args()
    select_config(args)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_product(args)


if __name__ == "__main__":
    main()
