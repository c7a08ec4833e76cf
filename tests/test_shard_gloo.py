"""N>1 path on CPU: two gloo ranks shard sequences (s mod world), each encodes its shard with the batch API of the
test-only emulator build, rank 0 gathers the streams in order and prints their digests, which must equal those of the
unmodified reference's streams."""
import hashlib
import os
import subprocess
import sys

import pytest

import dsvlibs as L

WORKER = r'''
import hashlib, importlib.util, os, sys
sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch.distributed as dist
import dsvlibs as L
spec = importlib.util.spec_from_file_location("shard", os.path.join(L.PKG, "shard.py"))
shard = importlib.util.module_from_spec(spec); spec.loader.exec_module(shard)
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
w, h, fmt, n, nseq = 64, 48, "420", 2, 3
cfg = L.make_cfg(w, h, fmt, gop=12)
mine = shard.my_shard(nseq, rank, world)
seqs = [L.synth_sequence(w, h, fmt, n, 70 + s, 0) for s in mine]
enc = L.BatchEncoder(L.emu(), cfg, 2)
streams = enc.encode(seqs, n) if seqs else []
enc.close()
allst = shard.gather_in_order(list(zip(mine, streams)), nseq, rank, world)
if rank == 0:
    for s in range(nseq):
        print("SHARD %d %s" % (s, hashlib.md5(allst[s]).hexdigest()))
    print("SHARD_OK")
dist.destroy_process_group()
'''


@pytest.fixture(scope="module")
def emu():
    subprocess.run(["make", "-s", "-C", L.PKG, "emu"], check=True, stdout=subprocess.DEVNULL)
    return L.emu()


def test_two_rank_shard_gather(tmp_path, emu, ref):
    script = tmp_path / "worker.py"
    script.write_text("ROOT = %r\n" % L.ROOT + WORKER)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29531", str(script)],
                       capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "SHARD_OK" in r.stdout
    got = dict(line.split()[1:] for line in r.stdout.splitlines() if line.startswith("SHARD "))
    w, h, fmt, n = 64, 48, "420", 2
    cfg = L.make_cfg(w, h, fmt, gop=12)
    for s in range(3):
        want, _, _ = ref.encode_sequence(cfg, L.synth_sequence(w, h, fmt, n, 70 + s, 0), n)
        assert got[str(s)] == hashlib.md5(want).hexdigest(), "sequence %d differs" % s
