"""GPU test of the sharded multi-GPU path of bench.py: one process per rank, each corrects its contiguous, length-balanced range
of ONE read set through the product's C ABI; the index goes from rank 0 to the others as one blob; results are reassembled in
input order in a shared host segment and hashed.  With two GPUs the ranks use NCCL and their own GPUs; on a one-GPU box they
share GPU 0 and coordinate through gloo (same code otherwise).  The gathered output must have the same sha256 as the one-rank
run, and every read must match the digests of the unmodified reference (tests/golden/mini.read_sha.npz)."""
import json
import os
import socket
import subprocess
import sys

import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _run_bench(world, extra=()):
    from longreadselfcorrect_b200 import api
    base = [sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "mini", "--gpus", str(world), "--steps", "1", "--warmup", "1", "--e2e-steps", "1",
            "--cli", "--no-cpu-baseline", "--batch-mbp", "1.0"] + list(extra)
    if world == 1:
        r = subprocess.run(base, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=420)
        assert r.returncode == 0, r.stderr[-1500:]
        return json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    port = _free_port()
    two_gpus = api.device_count() >= world
    procs = []
    for rank in range(world):
        env = dict(os.environ, RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE=str(world), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        cmd = list(base)
        if not two_gpus:
            env["PBSC_BENCH_SAME_DEVICE"] = "1"
            cmd += ["--backend", "gloo"]
        procs.append(subprocess.Popen(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True))
    # a rank that dies leaves the others waiting in a collective: watch all of them, kill the rest as soon as one fails
    import time
    t0 = time.time()
    while any(p.poll() is None for p in procs):
        if any(p.poll() not in (None, 0) for p in procs) or time.time() - t0 > 420:
            for p in procs:
                if p.poll() is None:
                    p.kill()
            break
        time.sleep(0.5)
    outs = [p.communicate() for p in procs]
    assert all(p.returncode == 0 for p in procs), [o[1][-1500:] for o in outs]
    return json.loads([l for l in outs[0][0].splitlines() if l.startswith("{")][-1])


def test_two_ranks_shard_the_product_path_and_reassemble_in_order(tmp_path):
    one = _run_bench(1, ("--dump-outputs", str(tmp_path / "dump")))
    two = _run_bench(2)
    for j in (one, two):
        p = j["parity_vs_reference"]
        assert p["identical"] and p["mismatches"] == 0 and p["reads_compared"] == p["reads_hashed"] == j["config"]["reads"], p
        assert j["scaling"] == "strong" and j["gpu_launches"] > 0
    assert one["parity_vs_reference"]["output_sha256"] == two["parity_vs_reference"]["output_sha256"]
    assert two["n_gpus"] == 2 and two["config"]["batches_per_rank"] >= 1
    # the shipped binary, driven by the same bench leg, writes the same records
    assert one["e2e_cli"]["output_sha256"] == one["parity_vs_reference"]["output_sha256"], one["e2e_cli"]
    # --dump-outputs: the last timed step's counters of the sampled reads and the pieces of a sub-sample, consistent with each other
    import numpy as np
    d = {f[:-4]: np.load(tmp_path / "dump" / f) for f in os.listdir(tmp_path / "dump")}
    ids, n = d["stats_read_ids"], one["config"]["reads"]
    assert ids.dtype == np.float64 and ids.size == min(n, 100_000) and np.all(np.diff(ids) > 0)
    assert all(d[k].shape == ids.shape for k in d if k.startswith("stats_"))
    pids, npc = d["pieces_read_ids"], d["pieces_per_read"]
    assert 0 < pids.size == npc.size and np.isin(pids, ids).all()
    at = np.searchsorted(ids, pids)
    assert np.array_equal(npc, d["stats_n_pieces"][at] * d["stats_merge"][at])      # a read that is not merged returns no piece
    assert d["piece_lengths"].size == npc.sum() and d["pieces_bases"].dtype == np.float32
    assert d["pieces_bases"].size == d["piece_lengths"].sum() and set(np.unique(d["pieces_bases"])) <= {65.0, 67.0, 71.0, 84.0}
    assert sum(a.nbytes for a in d.values()) <= 64 << 20
