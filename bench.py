#!/usr/bin/env python3
"""Benchmark of the `stride pbcorrect` hot path (seed discovery + FM extension + DP/MSA fallback) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg3|cfg2|cfg3s|cfg1|mini] [--nodp]
                    [--cli] [--extras] [--dump-outputs DIR]

One "step" = one pass of the hot path over the WHOLE read set of the workload.  The default workload is BASELINE.json
configs[2], the configuration its metric ("corrected Mbp/s at 1/2/4/8 B200") is quoted on: 12 Mb synthetic genome with
injected repeats, 100x simulated CLR reads (mean 8 kb, 1.24 Gbp), `-c 100 -g 10`, the reference's default options
(DP / multiple-alignment fallback on).  It fits one GPU.  `--workload cfg2` is configs[1] (4.6 Mb, 50x), also reported as a
sub-result of the line at N = 1 with --extras.

N > 1 (torchrun, one process per GPU): STRONG scaling of the product path.  Rank 0 simulates the reads and builds the index
once; the flat index travels to the other GPUs as one blob over NCCL (NVLink), the reads through /dev/shm.  Every rank takes
its contiguous, length-balanced range of the ONE read set (sharding.shard), cuts it into batches and runs them through the
lanes of its index (several batches in flight on separate streams).  No collective on the data path.
  value   total Mbp / max-over-ranks device time of a step (CUDA events), reads already resident in HBM
  e2e     the same through pbsc_correct_batch with HOST buffers: pinned H2D of the reads, D2H of the corrected pieces, every
          rank writing its results into one shared host segment in input order (the reassembly the reference does in
          SequenceProcessFramework.h:147-195); time = max over ranks of the wall clock between two barriers
  parity  every read of the gathered e2e output is hashed (parity.py) and compared with the digests the UNMODIFIED reference
          produced (tests/golden/<workload>.read_sha.npz); `output_sha256` identifies the whole output and must be the same
          at every N
  e2e_cli (--cli) the shipped binary, `pbcorrect --gpus N`, on a FASTA file (reader -> N GPU workers -> in-order writer)
`--impl reference` times the reference's own multithreaded CPU implementation (oracle/_ref/stride pbcorrect -t <cores>)
on a bounded sample of the same reads against the same index files, with the same options.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import re
import shutil
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True     # the tree may be read-only: nothing of this run is cached there

WORKLOADS = {
    # name: genome length, genome seed, coverage, mean read length, read seed, pbcorrect options
    "cfg2": dict(genome=4_600_000, gseed=2, cov=50, mean=8000, rseed=102, c=50, g=5,
                 desc="4.6 Mb synthetic genome, 50x simulated CLR reads (mean 8 kb, 13% error), -c 50 -g 5"),
    "cfg1": dict(genome=1_000_000, gseed=1, cov=30, mean=6000, rseed=101, c=30, g=5,
                 desc="1 Mb synthetic genome, 30x simulated CLR reads (mean 6 kb, 13% error), -c 30 -g 5"),
    # BASELINE.json configs[2] (12 Mb with injected repeats, 100x): 50 repeat families x 20 copies, 20 tandem arrays
    "cfg3": dict(genome=12_000_000, gseed=3, cov=100, mean=8000, rseed=103, c=100, g=10, repeat_families=50, tandem_arrays=20,
                 desc="12 Mb synthetic genome with injected repeats, 100x simulated CLR reads (mean 8 kb, 13% error), -c 100 -g 10"),
    # the same recipe at 1/6 of the size: a repeat-rich parity and capacity check that fits a short GPU slot
    "cfg3s": dict(genome=2_000_000, gseed=3, cov=100, mean=8000, rseed=103, c=100, g=10, repeat_families=8, tandem_arrays=4,
                  desc="2 Mb synthetic genome with injected repeats, 100x simulated CLR reads (mean 8 kb, 13% error), -c 100 -g 10"),
    # BASELINE.json configs[3]: 100 Mb genome, 40x: 4.0 G symbols with the sentinels, just inside the 32-bit positions of the index
    "cfg4": dict(genome=100_000_000, gseed=4, cov=40, mean=8000, rseed=104, c=40, g=100, sim="device",
                 desc="100 Mb synthetic genome, 40x simulated CLR reads (mean 8 kb, 13% error), -c 40 -g 100"),
    "mini": dict(genome=100_000, gseed=1, cov=30, mean=3000, rseed=101, c=30, g=5,
                 desc="100 kb synthetic genome, 30x simulated CLR reads (mean 3 kb), -c 30 -g 5"),
}
REF_STRIDE = os.path.join(ROOT, "oracle", "_ref", "stride")
ORACLE = os.path.join(ROOT, "oracle", "pbsc_oracle")
PBCORRECT = os.path.join(ROOT, "longreadselfcorrect_b200", "pbcorrect")
COUNT_LIB = os.path.join(ROOT, "longreadselfcorrect_b200", "libpbsc_count.so")


def log(*a):
    print("[bench]", *a, file=sys.stderr, flush=True)


def make_data(wl):
    from longreadselfcorrect_b200 import synth
    t = time.time()
    g = synth.make_genome(wl["genome"], wl["gseed"], repeat_families=wl.get("repeat_families", 0), tandem_arrays=wl.get("tandem_arrays", 0))
    if wl.get("sim") == "device":   # read sets numpy cannot simulate in one piece (config 4)
        codes, off = synth.simulate_reads_device(g, wl["cov"], wl["mean"], wl["rseed"])
    else:
        codes, off = synth.simulate_reads(g, wl["cov"], wl["mean"], wl["rseed"])
    log(f"simulated {off.size - 1} reads, {codes.size / 1e6:.1f} Mbp in {time.time() - t:.1f}s")
    return codes, off


def packed_ascii(codes, off):
    letters = np.frombuffer(b"ACGT", dtype=np.uint8)[codes]
    return np.ascontiguousarray(letters), off.astype(np.uint64)


class ClockSampler(threading.Thread):
    """nvidia-smi clocks and throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, gpu_index: int):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._halt = threading.Event()

    def run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._halt.is_set():
            try:
                r = subprocess.run(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                   stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=5)
                f = [x.strip() for x in r.stdout.strip().split(",")]
                if len(f) >= 6:
                    self.samples.append(float(f[0]))
                    self.max_mhz = float(f[1])
                    for nm, v in zip(names, f[2:6]):
                        if v.lower().startswith("active"):
                            self.reasons.add(nm)
            except Exception:
                pass
            self._halt.wait(0.2)

    def stop(self):
        self._halt.set()
        self.join(timeout=6)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def write_index_files(prefix, runs, n_reads):
    from longreadselfcorrect_b200 import bwt_build
    for ext in ("bwt", "rbwt"):
        r, nsym, nstr = runs[ext]
        bwt_build.write_bwt_file(f"{prefix}.{ext}", r, nstr, nsym)
    bwt_build.write_sai_file(prefix + ".sai", n_reads)


def write_fasta_ids(path, letters, off, ids):
    with open(path, "wb") as f:
        for i in ids:
            f.write(b">r%d\n" % i)
            f.write(letters[int(off[i]):int(off[i + 1])].tobytes())
            f.write(b"\n")


def run_reference(prefix, fa, wl, threads, outdir, nodp):
    """`stride pbcorrect -t T [--nodp]`; returns (seconds of the processing loop, wall seconds)."""
    t0 = time.time()
    r = subprocess.run([REF_STRIDE, "pbcorrect", "-t", str(threads), "-p", prefix, "-o", outdir, "-c", str(wl["c"]), "-g", str(wl["g"])]
                       + (["--nodp"] if nodp else []) + [fa], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    wall = time.time() - t0
    if r.returncode != 0:
        raise RuntimeError("reference failed: " + r.stderr[-500:])
    m = re.search(r"Processed \d+ sequences in ([0-9.]+)s", r.stderr)
    return (float(m.group(1)) if m else wall), wall


def oracle_rank_queries(prefix, fa, wl, threads, nodp):
    """Algorithmic work of the reference algorithm on a sample (instrumented oracle, SURVEY 8d): rank queries of the seed phase,
    of the walk constructor (E1: terminal intervals, query idmer / 5-mer trees) and of the level loop (E2-E12), separately; for
    the DP fallback the band cells filled, rows kept and LF steps."""
    with tempfile.TemporaryDirectory() as d:
        r = subprocess.run([ORACLE, "pbcorrect", "--threads", str(threads), "-p", prefix, "-o", os.path.join(d, "o"), "-c", str(wl["c"]),
                            "-g", str(wl["g"])] + (["--nodp"] if nodp else []) + [fa], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    m = re.search(r"rank queries (\d+) \(seed (\d+), extend (\d+)(?:: setup (\d+), walk loop (\d+))?\), walks (\d+)", r.stderr)
    if not m:
        return None
    out = {"total": int(m.group(1)), "seed": int(m.group(2)), "extend": int(m.group(3)), "walks": int(m.group(6))}
    if m.group(4) is not None:
        out["extend_setup"], out["extend_walk"] = int(m.group(4)), int(m.group(5))
    m = re.search(r"dp fallbacks (\d+), rows kept (\d+), band cells (\d+), LF steps (\d+)", r.stderr)
    if m:
        out.update({"dp_jobs": int(m.group(1)), "dp_rows_kept": int(m.group(2)), "dp_cells": int(m.group(3)), "dp_lf_steps": int(m.group(4))})
    return out


def sample_ids(n_reads, lengths, mbp, seed=20261018):
    """A seeded sample of reads spread over the whole set (NOT a prefix), about `mbp` Mbp; sorted ids."""
    rng = np.random.Generator(np.random.PCG64(seed))
    perm = rng.permutation(n_reads)
    cum = np.cumsum(lengths[perm])
    k = int(np.searchsorted(cum, mbp * 1e6)) + 1
    return np.sort(perm[: max(1, min(k, n_reads))])


# ---------------------------------------------------------------------------------------------------------------------
# reference arm (CPU)
# ---------------------------------------------------------------------------------------------------------------------
def reference_arm(args, wl, metric):
    cores = os.cpu_count() or 1
    codes, off = make_data(wl)
    from longreadselfcorrect_b200 import bwt_build
    total_mbp = codes.size / 1e6
    n_reads = off.size - 1
    lengths = np.diff(off)
    # The reference pays tens of seconds per process to load a 1.2 Gbp index, so the W + K steps are consecutive slices of ONE
    # process run: a seeded sample of (W + K) x ~S Mbp spread over the whole read set; ms_per_step = its processing-loop time
    # (the reference's own "Processed N sequences in Xs" line, index load excluded) / (W + K).
    slices = args.warmup + args.steps
    per_step = args.cpu_sample_mbp or max(0.4, min(total_mbp / slices, 0.035 * cores * 12))
    ids = sample_ids(n_reads, lengths, per_step * slices)
    sample_mbp = float(lengths[ids].sum()) / 1e6
    letters = np.frombuffer(b"ACGT", dtype=np.uint8)[codes]
    with tempfile.TemporaryDirectory(dir="/dev/shm" if os.path.isdir("/dev/shm") else None) as d:
        prefix = os.path.join(d, "idx")
        bwt_build.build_index_files(prefix, codes, off)
        fa = os.path.join(d, "sample.fa")
        write_fasta_ids(fa, letters, off, ids)
        secs, wall = run_reference(prefix, fa, wl, cores, os.path.join(d, "out"), args.nodp)
        log(f"reference: {ids.size} reads ({sample_mbp:.1f} Mbp) in {secs:.2f}s processing ({wall:.1f}s wall incl. index load), {cores} threads")
    ms = 1000 * secs / slices
    v = sample_mbp / secs
    sample_desc = (f"seeded sample of {ids.size} reads spread over the whole set ({sample_mbp:.1f} Mbp of {total_mbp:.1f}) against the full index; "
                   f"the {slices} steps are consecutive slices of one process run (index load excluded)")
    print(json.dumps({
        "impl": "reference", "metric": metric, "value": v, "unit": "Mbp/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "int64+f64", "data": "synthetic",
        "config": {"workload": wl["desc"], "sample": sample_desc, "threads": cores},
        "cpu_baseline": {"value": v, "unit": "Mbp/s", "cores": cores, "kind": "reference", "sample": sample_desc},
        "e2e": {"value": v, "unit": "Mbp/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))
    return 0


# ---------------------------------------------------------------------------------------------------------------------
# our arm (GPU)
# ---------------------------------------------------------------------------------------------------------------------
class Shard:
    """One rank's contiguous range of the read set, cut into batches."""

    def __init__(self, letters, off, begin, end, batch_mbp):
        from longreadselfcorrect_b200 import sharding
        self.begin, self.end = begin, end
        o = off[begin:end + 1]
        self.bases = int(o[-1] - o[0])
        nb = max(1, int(np.ceil(self.bases / (batch_mbp * 1e6))))
        self.batches = []     # (first read id, ascii bytes, offsets)
        for b0, b1 in sharding.balanced_ranges(np.diff(o), nb):
            if b1 <= b0:
                continue
            oo = o[b0:b1 + 1]
            self.batches.append((begin + b0, np.ascontiguousarray(letters[int(oo[0]):int(oo[-1])]), (oo - oo[0]).astype(np.uint64)))


def run_threads(n_threads, n_items, fn):
    """fn(i) for i in range(n_items) from n_threads host threads (the library releases the GIL inside its calls)."""
    if n_threads <= 1 or n_items <= 1:
        for i in range(n_items):
            fn(i)
        return
    nxt, lock, errs = [0], threading.Lock(), []

    def work():
        while True:
            with lock:
                i = nxt[0]
                nxt[0] += 1
            if i >= n_items or errs:
                return
            try:
                fn(i)
            except BaseException as e:   # noqa: BLE001
                errs.append(e)
    th = [threading.Thread(target=work) for _ in range(min(n_threads, n_items))]
    for t in th:
        t.start()
    for t in th:
        t.join()
    if errs:
        raise errs[0]


TIMING_KEYS = ("seed_ms", "extend_ms", "dp_ms", "walk_ms", "walk_launches", "dp_jobs", "dp_rows", "kernel_launches", "seed_pairs")

# --dump-outputs: one seeded sample of the reads, drawn from the input lengths only, so that two builds dump the same reads;
# counters of up to DUMP_READS reads and the corrected pieces of the first ~DUMP_PIECE_MBP input Mbp of the same permutation
# (config 3: 100 k reads and ~4 M bases, ~30 MB of .npy files)
DUMP_SEED = 20261020
DUMP_READS = 100_000
DUMP_PIECE_MBP = 4.0


def dump_outputs(path, shard, batches, lengths):
    """What the timed path returned for the reads of its last step (Batch.fetch: corrected pieces, their offsets, the first
    piece of every read, the per-read counters), for the seeded sample above, as float64 .npy files (the bases as float32)."""
    from longreadselfcorrect_b200 import api
    perm = np.random.Generator(np.random.PCG64(DUMP_SEED)).permutation(lengths.size)
    stat_ids = np.sort(perm[:DUMP_READS])
    piece_ids = np.sort(perm[:int(np.searchsorted(np.cumsum(lengths[perm]), DUMP_PIECE_MBP * 1e6)) + 1])
    stats = np.zeros(stat_ids.size, dtype=api.STATS_DTYPE)
    n_pieces, piece_len, bases = [], [], []
    for (f, _a, o), bt in zip(shard.batches, batches):
        n = o.size - 1
        out, poff, first, st = bt.fetch()
        sel = stat_ids[(stat_ids >= f) & (stat_ids < f + n)]
        stats[np.searchsorted(stat_ids, sel)] = st[sel - f]
        for r in piece_ids[(piece_ids >= f) & (piece_ids < f + n)] - f:
            p0, p1 = int(first[r]), int(first[r + 1])
            n_pieces.append(p1 - p0)
            piece_len.extend(int(poff[j + 1] - poff[j]) for j in range(p0, p1))
            bases.append(out[int(poff[p0]):int(poff[p1])].copy())
    os.makedirs(path, exist_ok=True)
    arrays = {"stats_read_ids": stat_ids, "pieces_read_ids": piece_ids, "pieces_per_read": n_pieces, "piece_lengths": piece_len}
    arrays.update({f"stats_{k}": stats[k] for k in api.STATS_DTYPE.names})
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), np.asarray(a, dtype=np.float64))
    np.save(os.path.join(path, "pieces_bases.npy"), np.concatenate(bases).astype(np.float32) if bases else np.zeros(0, np.float32))
    log(f"outputs of the last timed step: {stat_ids.size} reads' counters, {piece_ids.size} reads' pieces "
        f"({sum(len(b) for b in bases)} bases) in {path}")


def ours(args, wl, metric):
    import torch
    from longreadselfcorrect_b200 import api, bwt_build, parity, sharding
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cores = os.cpu_count() or 1
    assert torch.cuda.is_available(), "bench.py needs a CUDA device: the hot path has no CPU fallback"
    assert not (args.dump_outputs and world > 1), "--dump-outputs needs one rank: the outputs of a step are spread over the ranks' shards"
    # --backend gloo: the same multi-rank code without NCCL (control traffic through gloo on CPU tensors), for boxes where the
    # ranks have to share one GPU (tests); PBSC_BENCH_SAME_DEVICE=1 puts every rank on GPU 0
    if os.environ.get("PBSC_BENCH_SAME_DEVICE") == "1":
        local_rank = 0
    torch.cuda.set_device(local_rank)
    dist = None
    cdev = "cuda" if args.backend == "nccl" else "cpu"
    if world > 1:
        import torch.distributed as dist
        if args.backend == "nccl":
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        else:
            dist.init_process_group("gloo")
        # a CPU-side group for waiting without touching the GPUs: an NCCL barrier is a kernel that spins on every waiting rank's
        # GPU, and during the e2e_cli leg those GPUs belong to the pbcorrect process (measured: 6.5 s instead of 2.7 s)
        cpu_group = dist.new_group(backend="gloo") if args.backend == "nccl" else None

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(vals):
        if dist is None:
            return [float(v) for v in vals]
        tt = torch.tensor(list(vals), device=cdev, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return [float(x) for x in tt]

    # ---- the ONE read set: simulated by rank 0, shared through /dev/shm ----
    shm = os.path.join("/dev/shm" if os.path.isdir("/dev/shm") else tempfile.gettempdir(),
                       f"pbsc_bench_{os.environ.get('MASTER_PORT', '0')}_{os.environ.get('TORCHELASTIC_RUN_ID', str(os.getppid()) if world > 1 else str(os.getpid()))}")
    runs = None
    if rank == 0:
        shutil.rmtree(shm, ignore_errors=True)
        os.makedirs(shm)
        codes, off = make_data(wl)
        letters, off = packed_ascii(codes, off)
        if world > 1:
            np.save(os.path.join(shm, "letters.npy"), letters)
            np.save(os.path.join(shm, "off.npy"), off)
    barrier()
    if rank != 0:
        letters = np.load(os.path.join(shm, "letters.npy"), mmap_mode="r")
        off = np.load(os.path.join(shm, "off.npy"))
    n_reads = off.size - 1
    lengths = np.diff(off.astype(np.int64))
    total_mbp = float(off[-1]) / 1e6

    # ---- the index: built once on rank 0, broadcast as one blob over NCCL ----
    t = time.time()
    if rank == 0:
        # `stride index` on the GPU (pbsc_build.cu, SURVEY.md 8f-2): the same bytes the reference's ropebwt2 path writes
        runs = {}
        for ext, rev in (("bwt", False), ("rbwt", True)):
            r, nsym, _ = api.build_bwt((letters, off), reverse=rev, device=local_rank)
            runs[ext] = (r, nsym, n_reads)
        bwt_s = time.time() - t
        log(f"rank 0: BWT + RBWT of {total_mbp:.1f} Mbp built by pbsc_build_bwt in {bwt_s:.1f}s (index construction, not part of the timed step)")
        t = time.time()
        idx = api.Index.from_runs(runs["bwt"][0], runs["bwt"][1], n_reads, runs["rbwt"][0], runs["rbwt"][1], n_reads, device=local_rank)
        if args.k0:
            idx.build_prefix_table(args.k0)
        del codes
    index_s = time.time() - t
    bcast_s = 0.0
    if world > 1:
        t = time.time()
        nb = torch.tensor([idx.blob_size() if rank == 0 else 0], device=cdev, dtype=torch.int64)
        dist.broadcast(nb, 0)
        blob = torch.empty(int(nb[0]), dtype=torch.uint8, device="cuda")
        if rank == 0:
            idx.export_blob(blob.data_ptr(), blob.numel())
        if args.backend == "nccl":
            dist.broadcast(blob, 0)          # NVLink / NVSwitch: the one exchange of the job, off the data path
            torch.cuda.synchronize()
            if rank != 0:
                idx = api.Index.import_blob(blob.data_ptr(), blob.numel(), local_rank, local_rank)
        else:
            hblob = blob.cpu()
            dist.broadcast(hblob, 0)
            if rank != 0:
                idx = api.Index.import_blob(hblob.data_ptr(), hblob.numel(), -1, local_rank)
            del hblob
        del blob
        torch.cuda.empty_cache()
        bcast_s = time.time() - t
    idx.set_lanes(args.lanes)
    log(f"rank {rank}: index on device ({idx.device_bytes() / 1e9:.2f} GB; decode + prefix table {index_s:.1f}s on rank 0, NCCL broadcast {bcast_s:.2f}s), {args.lanes} lanes")
    params = api.Params.make(coverage=wl["c"], genome=wl["g"], no_dp=args.nodp)

    # ---- this rank's shard of the read set ----
    b_, e_ = sharding.balanced_ranges(lengths, world)[rank]
    shard = Shard(letters, off, b_, e_, args.batch_mbp)
    nbt = len(shard.batches)
    log(f"rank {rank}: reads [{b_}, {e_}) = {shard.bases / 1e6:.1f} Mbp in {nbt} batch(es)")

    # ---- value: reads resident on the device (batches uploaded before the timed region when they all fit), kernels only ----
    # a batch that is not running holds only its reads (one byte per base) and, after a run, its results: all of them stay resident
    resident_ok = True
    resident = [api.Batch(idx, params, packed=(a, o)) for (_f, a, o) in shard.batches]
    tm_lock = threading.Lock()

    def run_step():
        """one pass over this rank's batches through the lanes; returns (device ms between CUDA events, summed phase counters)"""
        acc = {k: 0.0 for k in TIMING_KEYS}

        def one(i):
            if resident is not None:
                resident[i].run()
                tm = api.last_timing()
            else:
                f, a, o = shard.batches[i]
                bt = api.Batch(idx, params, packed=(a, o))
                bt.run()
                tm = api.last_timing()
                bt.close()
            with tm_lock:
                for k in TIMING_KEYS:
                    acc[k] += tm[k]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        run_threads(args.lanes, nbt, one)
        torch.cuda.synchronize()
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1), acc

    for _ in range(args.warmup):
        run_step()
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    step_ms, phases = [], []
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ms, acc = run_step()
        step_ms.append(ms)
        phases.append(acc)
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1000
    clocks = sampler.stop()
    dev_ms, wall_ms = allmax([float(np.sum(step_ms)), wall_ms])
    ms_per_step = dev_ms / args.steps
    value = total_mbp / (ms_per_step / 1000)
    ph = {k: float(np.mean([p[k] for p in phases])) for k in TIMING_KEYS}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, shard, resident, lengths)
    if resident is not None:
        for bt in resident:
            bt.close()
    resident = None
    api.lib().pbsc_trim(local_rank)

    # ---- e2e: host buffers in, corrected pieces out, through pbsc_correct_batch.  Reads sit in pinned host memory; every rank
    #      writes its results (pieces, offsets, counters) straight into ITS region of one shared host segment, in input order,
    #      so after the closing barrier rank 0 holds the reassembled output of the whole read set. ----
    pin_in = [(api.pinned_copy(a), api.pinned_copy(o)) for (_f, a, o) in shard.batches]
    seg = []   # per batch: dict of numpy views into this rank's shared file
    layout = []
    pos = 0
    for (f, a, o) in shard.batches:
        n = o.size - 1
        cap = int(a.size * 1.25) + (1 << 16)
        ent = {"first_id": f, "n": n, "out": (pos, cap)}
        pos += (cap + 255) // 256 * 256
        ent["poff"] = (pos, (n + 2) * 8); pos += (n + 2) * 8
        ent["first"] = (pos, (n + 1) * 8); pos += (n + 1) * 8
        ent["stats"] = (pos, max(n, 1) * api.STATS_DTYPE.itemsize); pos += (max(n, 1) * api.STATS_DTYPE.itemsize + 255) // 256 * 256
        layout.append(ent)
    seg_path = os.path.join(shm, f"out_rank{rank}.bin")
    with open(seg_path, "wb") as fh:
        fh.truncate(max(pos, 4096))
    mm = np.memmap(seg_path, dtype=np.uint8, mode="r+")
    mm[:] = 0              # touch every page before it is page-locked
    api.host_register(mm)

    def views(m, ent):
        o0, oc = ent["out"]; p0, pc = ent["poff"]; f0, fc = ent["first"]; s0, sc = ent["stats"]
        return (m[o0:o0 + oc], m[p0:p0 + pc].view(np.uint64), m[f0:f0 + fc].view(np.uint64), m[s0:s0 + sc].view(api.STATS_DTYPE))
    seg = [views(mm, ent) for ent in layout]

    def e2e_step():
        def one(i):
            idx.correct_reads(params, packed=pin_in[i], out_bufs=seg[i])
        run_threads(args.lanes + 1, nbt, one)   # one thread more than lanes: its upload / fetch overlaps the others' kernels
        torch.cuda.synchronize()

    e2e_times = []
    for i in range(args.e2e_steps + 1):
        barrier()
        t0 = time.perf_counter()
        e2e_step()
        barrier()
        if i > 0:
            e2e_times.append((time.perf_counter() - t0) * 1000)
    e2e_ms = allmax([float(np.mean(e2e_times)) if e2e_times else float("nan")])[0]
    e2e_value = total_mbp / (e2e_ms / 1000)
    h2d_bytes = int(sum(a.nbytes + o.nbytes for a, o in pin_in))
    d2h_local = 0
    for (out, poff, first, stats), ent in zip(seg, layout):
        n = ent["n"]
        d2h_local += int(poff[int(first[n])]) + n * api.STATS_DTYPE.itemsize + 16 * n
    if dist is not None:
        tt = torch.tensor([h2d_bytes, d2h_local], device=cdev, dtype=torch.int64)
        dist.all_reduce(tt)
        h2d_bytes, d2h_bytes = int(tt[0]), int(tt[1])
        lay_all = [None] * world
        dist.all_gather_object(lay_all, layout)
    else:
        d2h_bytes, lay_all = d2h_local, [layout]
    api.host_unregister(mm)
    mm.flush()
    barrier()

    # ---- parity over the WHOLE gathered output (rank 0 reads every rank's region of the shared segment) ----
    par = None
    walks = fm = dpn = 0
    if rank == 0:
        t = time.time()
        dig = np.zeros((n_reads, 8), dtype=np.uint8)
        for r in range(world):
            m = mm if r == 0 else np.memmap(os.path.join(shm, f"out_rank{r}.bin"), dtype=np.uint8, mode="r")
            for ent in lay_all[r]:
                out, poff, first, stats = views(m, ent)
                f, n = ent["first_id"], ent["n"]
                st = stats[:n]
                dig[f:f + n] = parity.result_digests(out, poff, first, st, letters[int(off[f]):int(off[f + n])], off[f:f + n + 1] - off[f], first_read_id=f)
                mg = st[st["merge"] == 1]
                walks += int(mg["total_walk_num"].sum()); fm += int(mg["fm_num"].sum()); dpn += int(mg["dp_num"].sum())
        par = {"output_sha256": parity.output_sha256(dig), "reads_hashed": int(n_reads),
               "what": "sha256 over the per-read record digests (parity.py) of the gathered e2e output of the last timed step, input order"}
        cmp_ = parity.compare_with_golden(args.workload + ("_nodp" if args.nodp else ""), dig)
        if cmp_:
            par.update(cmp_)
        log(f"parity: {par} ({time.time() - t:.1f}s)")
    del seg, mm

    # ---- e2e_cli: the shipped binary on a FASTA file with the index files of `stride index`, all N GPUs, one process ----
    cli = None
    if args.cli and os.path.exists(PBCORRECT):
        idx.close()
        api.lib().pbsc_trim(local_rank)
        torch.cuda.empty_cache()
        barrier()
        if rank == 0:
            try:
                cli = run_cli(args, wl, shm, letters, off, runs, n_reads, total_mbp, world, cores, parity)
            except Exception as e:   # measurement leg only
                cli = {"error": str(e)[-300:]}
            log(f"e2e_cli: {cli}")
        if dist is not None:
            dist.barrier(group=cpu_group)      # the other ranks wait on the CPU: their GPUs are the binary's
        idx = None

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return 0

    line = {
        "metric": metric, "value": value, "unit": "Mbp/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "int64+f64", "data": "synthetic",
        "config": {"workload": wl["desc"], "reads": int(n_reads), "mbp": total_mbp, "walks": walks, "fm_success": fm, "dp_success": dpn,
                   "prefix_k0": args.k0, "lanes": args.lanes, "batch_mbp": args.batch_mbp, "batches_per_rank": nbt,
                   "bwt_build_s": bwt_s if rank == 0 else None, "bwt_builder": "pbsc_build_bwt (pbsc_build.cu)", "index_build_s": index_s, "index_broadcast_s": bcast_s,
                   "l2": "rank tables + prefix table exceed the 126 MB L2; no explicit flush",
                   "sharding": "one read set; contiguous length-balanced range per rank; index built on rank 0 and broadcast as one blob over NCCL; "
                               "results reassembled in input order in a shared host segment; no collective on the data path",
                   "reads_resident_before_timed_region": bool(resident_ok),
                   "wall_ms_per_step": wall_ms / args.steps},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "Mbp/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes, "ms_per_step": e2e_ms,
                "steps": len(e2e_times)},
        "gpu_launches": int(ph["kernel_launches"]) * args.steps,
        "parity_vs_reference": par,
        "e2e_cli": cli,
        "phases_ms_rank0": {k: ph[k] for k in ("seed_ms", "extend_ms", "walk_ms", "dp_ms")},
    }

    # ---- single-GPU extras: CPU baseline, algorithmic and issued rank queries, roofline, config 2 / --nodp / FM microbench ----
    if world == 1:
        extras_single_gpu(args, wl, line, letters, off, runs, n_reads, total_mbp, lengths, ph, walks, cores, local_rank, dig)
    else:
        line["roofline"] = roofline_from_committed(args, ph, walks * shard.bases / max(1.0, total_mbp * 1e6), total_mbp)
        line["cpu_baseline"] = None
    print(json.dumps(line))
    shutil.rmtree(shm, ignore_errors=True)
    if dist is not None:
        dist.destroy_process_group()
    return 0


def run_cli(args, wl, shm, letters, off, runs, n_reads, total_mbp, world, cores, parity):
    """`pbcorrect --gpus N` on files: FASTA of the whole read set + PREFIX.bwt/.rbwt/.sai; returns throughputs and the parity of
    the files it wrote."""
    prefix = os.path.join(shm, "idx")
    write_index_files(prefix, runs, n_reads)
    fa = os.path.join(shm, "reads.fa")
    write_fasta_ids(fa, letters, off, range(n_reads))
    out = os.path.join(shm, "cli_out")
    res = {}
    for attempt in ("cold (decodes PREFIX.bwt/.rbwt, writes PREFIX.fmg)", "warm (PREFIX.fmg)"):
        shutil.rmtree(out, ignore_errors=True)
        t0 = time.time()
        r = subprocess.run([PBCORRECT, "pbcorrect", "-t", str(min(cores, 16)), "--gpus", str(world), "-p", prefix, "-o", out, "-c", str(wl["c"]), "-g", str(wl["g"]),
                            "--batch-mbp", str(args.batch_mbp), "--lanes", str(args.lanes)] + (["--nodp"] if args.nodp else []) + [fa],
                           stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
        wall = time.time() - t0
        if r.returncode != 0:
            raise RuntimeError("pbcorrect failed: " + r.stderr[-400:])
        m = re.search(r"Processed \d+ sequences in ([0-9.]+)s", r.stderr)
        secs = float(m.group(1)) if m else wall
        m2 = re.search(r"index to \d+ GPU\(s\)\] wall clock: ([0-9.]+)s", r.stderr)
        key = "cold" if attempt.startswith("cold") else "warm"
        res[key] = {"processing_s": secs, "wall_s": wall, "index_load_s": float(m2.group(1)) if m2 else None, "what": attempt}
    dg = parity.fasta_digests(os.path.join(out, "correct.fa"), os.path.join(out, "discard.fa"))
    dig = np.zeros((n_reads, 8), dtype=np.uint8)
    for i in range(n_reads):
        if i in dg:
            dig[i] = np.frombuffer(dg[i], dtype=np.uint8)
    secs = res["warm"]["processing_s"]
    return {"value": total_mbp / secs, "unit": "Mbp/s", "gpus": world,
            "what": "pbcorrect --gpus N: FASTA parse -> batches -> lanes of N GPUs -> in-order writer of correct.fa / discard.fa; Mbp of input / the "
                    "binary's own processing time (index load reported separately, as the reference does)",
            "processing_s": secs, "wall_s_incl_index_load": res["warm"]["wall_s"], "index_load_s_fmg": res["warm"]["index_load_s"],
            "index_load_s_bwt": res["cold"]["index_load_s"], "records": len(dg), "output_sha256": parity.output_sha256(dig)}


def roofline_from_committed(args, ph, walks, total_mbp):
    """N > 1 (no CPU legs): per-unit algorithmic work from the committed oracle measurement (profiles/algorithmic.json)."""
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    roof = {"bound": "hbm", "kernel": "walk_levels_kernel", "achieved": None, "peak": peak, "unit": "GB/s", "frac": None, "traffic": None,
            "peak_source": "MEASURED_PEAKS.json hbm_gbs (streaming copy)" if peaks else "fallback 6650 GB/s (B200_PROFILING.md)",
            "kernel_ms_rank0": ph["walk_ms"], "note": "rank 0's share of the step; algorithmic counts from profiles/algorithmic.json"}
    try:
        c = json.load(open(os.path.join(ROOT, "profiles", "algorithmic.json"))).get(args.workload + ("_nodp" if args.nodp else ""))
        if c and c.get("walk_loop_rank_queries_per_walk") and ph["walk_ms"] > 0:
            b = c["walk_loop_rank_queries_per_walk"] * walks * 32.0      # `walks`: the reference's walks of rank 0's share of the reads
            roof["achieved"] = b / (ph["walk_ms"] / 1000) / 1e9
            roof["frac"] = roof["achieved"] / peak
    except Exception:
        pass
    return roof


def count_issued(args, wl, letters, off, runs, n_reads, ids, local_rank):
    """Issued 32-byte rank sectors per kernel family, from the PBSC_COUNT_OCC build of the library run in a child process on the
    same sample the oracle counted (tools/count_occ.py)."""
    if not os.path.exists(COUNT_LIB):
        return None
    with tempfile.TemporaryDirectory(dir="/dev/shm" if os.path.isdir("/dev/shm") else None) as d:
        prefix = os.path.join(d, "idx")
        write_index_files(prefix, runs, n_reads)
        fa = os.path.join(d, "s.fa")
        write_fasta_ids(fa, letters, off, ids)
        env = dict(os.environ, PBSC_LIB=COUNT_LIB)
        r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "count_occ.py"), prefix, fa, str(wl["c"]), str(wl["g"]), str(args.k0), str(local_rank)]
                           + (["--nodp"] if args.nodp else []), env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    for l in r.stdout.splitlines():
        if l.startswith("{"):
            return json.loads(l)
    log("issued-sector count failed:", r.stderr[-300:])
    return None


def extras_single_gpu(args, wl, line, letters, off, runs, n_reads, total_mbp, lengths, ph, walks, cores, local_rank, dig=None):
    from longreadselfcorrect_b200 import api
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    cpu = alg = issued = None
    if not args.no_cpu_baseline and os.path.exists(REF_STRIDE):
        # bounded: ~0.03 Mbp/s/core (repeat-rich, DP fallback on) x cores x ~15 s, as a seeded sample spread over the whole set
        smbp = args.cpu_sample_mbp or min(total_mbp, max(0.5, 0.03 * cores * 15))
        ids = sample_ids(n_reads, lengths, smbp)
        smbp = float(lengths[ids].sum()) / 1e6
        with tempfile.TemporaryDirectory(dir="/dev/shm" if os.path.isdir("/dev/shm") else None) as d:
            prefix = os.path.join(d, "idx")
            write_index_files(prefix, runs, n_reads)
            fa = os.path.join(d, "sample.fa")
            write_fasta_ids(fa, letters, off, ids)
            secs, wall = run_reference(prefix, fa, wl, cores, os.path.join(d, "out"), args.nodp)
            log(f"reference CPU baseline: {smbp:.1f} Mbp in {secs:.2f}s with {cores} threads")
            sdesc = f"seeded sample of {ids.size} reads spread over the whole set ({smbp:.1f} Mbp of {total_mbp:.1f}) against the full index, stride pbcorrect -t {cores}" + (" --nodp" if args.nodp else "")
            cpu = {"value": smbp / secs, "unit": "Mbp/s", "cores": cores, "kind": "reference", "sample": sdesc}
            # live parity on exactly these reads: the records the unmodified reference just wrote against the timed GPU output
            if dig is not None and isinstance(line.get("parity_vs_reference"), dict):
                from longreadselfcorrect_b200 import parity
                ref = parity.fasta_digests(os.path.join(d, "out", "correct.fa"), os.path.join(d, "out", "discard.fa"))
                same = sum(1 for i in ids if int(i) in ref and bytes(ref[int(i)]) == bytes(dig[int(i)].tobytes()))
                line["parity_vs_reference"]["live_sample"] = {"reads": int(ids.size), "identical_to_reference": int(same),
                                                              "what": "the CPU baseline's reads: records written by oracle/_ref/stride pbcorrect against the full index, compared with the timed GPU output"}
                log(f"live parity: {same} of {ids.size} sampled reads identical to the reference")
            # live parity of exactly these reads: what the reference just wrote against the digests of the timed GPU output is
            # covered by parity_vs_reference when a golden exists; here the reference's records are hashed and kept
            if os.path.exists(ORACLE) and not args.no_oracle_count:
                small_ids = ids[: max(1, int(np.searchsorted(np.cumsum(lengths[ids]), min(smbp, 3.0) * 1e6)))]
                fa2 = os.path.join(d, "alg.fa")
                write_fasta_ids(fa2, letters, off, small_ids)
                alg = oracle_rank_queries(prefix, fa2, wl, min(cores, 32), args.nodp)
                if alg:
                    alg["sample_bases"] = int(lengths[small_ids].sum())
                issued = count_issued(args, wl, letters, off, runs, n_reads, small_ids, local_rank)
    line["cpu_baseline"] = cpu
    try:
        sector_peak = api.random_sector_peak(2_400_000_000, local_rank)
    except Exception as e:   # measurement aid only
        log("random-sector peak not measured:", e)
        sector_peak = None
    traffic = None
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        traffic = tr.get(args.workload + ("_nodp" if args.nodp else ""), {}).get("walk_levels_kernel")
    except Exception:
        pass
    walk_ms = ph["walk_ms"]
    roof = {"bound": "hbm", "kernel": "walk_levels_kernel", "achieved": None, "peak": peak, "unit": "GB/s", "frac": None, "traffic": traffic,
            "peak_source": "MEASURED_PEAKS.json hbm_gbs (streaming copy)" if peaks else "fallback 6650 GB/s (B200_PROFILING.md)",
            "kernel_ms": walk_ms, "kernel_launches_per_step": int(ph["walk_launches"]), "extend_phase_ms": ph["extend_ms"], "seed_phase_ms": ph["seed_ms"],
            "dp_fallback_ms": ph["dp_ms"], "walks_per_step": ph["seed_pairs"],
            "scope": "algorithmic bytes = rank queries of the reference's LEVEL LOOP only (extendOverlap, LongReadCorrectByOverlap.cpp:155-211; the "
                     "constructor's searches are counted apart as extend_setup) x 32 B, for the walks the kernel ran in the step, / the CUDA-event time "
                     "of walk_levels_kernel's own launches"}
    if not (alg and alg.get("walks")):
        try:
            c = json.load(open(os.path.join(ROOT, "profiles", "algorithmic.json"))).get(args.workload + ("_nodp" if args.nodp else ""))
            if c and c.get("walk_loop_rank_queries_per_walk"):
                alg = {"walks": 1.0, "extend_walk": c["walk_loop_rank_queries_per_walk"], "extend_setup": c.get("setup_rank_queries_per_walk", 0.0),
                       "extend": c["walk_loop_rank_queries_per_walk"] + c.get("setup_rank_queries_per_walk", 0.0),
                       "seed": c["seed_rank_queries_per_read_base"], "sample_bases": 1.0, "source": "profiles/algorithmic.json"}
        except Exception:
            pass
    if alg and alg.get("walks") and walk_ms > 0:
        loop_q = alg.get("extend_walk", alg["extend"]) / alg["walks"]
        # the kernel walks more pairs than the reference (speculative tasks that are re-walked): the algorithmic count uses the
        # reference's number of walks of the step, i.e. what had to be computed
        ref_walks = walks
        alg_bytes = loop_q * ref_walks * 32.0
        roof["achieved"] = alg_bytes / (walk_ms / 1000) / 1e9
        roof["frac"] = roof["achieved"] / peak
        roof["algorithmic_bytes_per_step"] = alg_bytes
        roof["algorithmic_rank_queries_per_walk_level_loop"] = loop_q
        roof["algorithmic_rank_queries_per_walk_constructor"] = alg.get("extend_setup", 0) / alg["walks"]
        roof["algorithmic_rank_queries_per_read_base_seed_phase"] = alg["seed"] / alg["sample_bases"]
        roof["seed_phase_algorithmic_GBs"] = alg["seed"] / alg["sample_bases"] * total_mbp * 1e6 * 32.0 / (ph["seed_ms"] / 1000) / 1e9
        roof["algorithmic_source"] = alg.get("source", "instrumented oracle (oracle/pbsc_oracle) on a sample of the same reads, this run")
        if issued and issued.get("walks"):
            per_walk = issued["walk"] / issued["walks"]
            isec = per_walk * ph["seed_pairs"]
            roof["issued_sectors_per_walk_level_loop"] = per_walk
            roof["issued_sectors_per_step_level_loop"] = isec
            roof["issued_GBs"] = isec * 32.0 / (walk_ms / 1000) / 1e9
            roof["issued"] = {k: issued[k] for k in ("seed", "setup", "walk", "dp", "walks", "bases") if k in issued}
            roof["issued_source"] = "libpbsc_count.so (-DPBSC_COUNT_OCC build of the same kernels) on the oracle's sample, per-kernel-family counters"
            if sector_peak:
                roof["random_sector_peak"] = sector_peak
                roof["frac_of_random_sector_peak"] = roof["issued_GBs"] / sector_peak
        elif sector_peak:
            roof["random_sector_peak"] = sector_peak
        if alg.get("dp_jobs"):
            cells = alg["dp_cells"] / alg["dp_jobs"] * ph["dp_jobs"]
            roof["dp_fallback"] = {"jobs_per_step": ph["dp_jobs"], "rows_aligned_per_step": ph["dp_rows"], "band_cells_per_step": cells,
                                   "Gcells_per_s": cells / (ph["dp_ms"] / 1000) / 1e9 if ph["dp_ms"] > 0 else None}
    line["roofline"] = roof
    if args.extras:
        line["sub_results"] = sub_results(args, local_rank)


def sub_results(args, local_rank):
    """The rest of the BASELINE metric in the same driver-visible line: config 2 (default options and --nodp) and the FM
    backward-search microbenchmark (config 5), each measured in a child process (fresh memory, bounded time)."""
    res = {}
    py = sys.executable
    base = [py, os.path.abspath(__file__), "--no-cpu-baseline", "--steps", str(args.steps), "--warmup", str(args.warmup)]
    env = dict(os.environ, PYTHONDONTWRITEBYTECODE="1")    # the children import modules of the tree, which must stay as build() left it
    for name, extra in (("cfg2_default_options", ["--workload", "cfg2"]), ("cfg2_nodp", ["--workload", "cfg2", "--nodp"])):
        if args.workload == "cfg2" and not args.nodp and name == "cfg2_default_options":
            continue
        try:
            r = subprocess.run(base + extra, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900, env=env)
            j = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
            res[name] = {"value": j["value"], "unit": j["unit"], "ms_per_step": j["ms_per_step"], "e2e": j["e2e"], "config": j["config"]["workload"],
                         "parity_vs_reference": j.get("parity_vs_reference"), "roofline": j.get("roofline"), "phases_ms": j.get("phases_ms_rank0")}
        except Exception as e:
            res[name] = {"error": str(e)[-200:]}
    try:
        # index construction (SURVEY.md 8f-2): both strands of config 2 by pbsc_build_bwt; the reference's `stride index` on a 1 Mbp sample
        r = subprocess.run([py, os.path.join(ROOT, "tools", "index_bench.py"), "--json", "--workload", "cfg2", "--skip-torch", "--reference-mbp", "1"],
                           stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600, env=env)
        res["index_build_cfg2"] = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    except Exception as e:
        res["index_build_cfg2"] = {"error": str(e)[-200:]}
    try:
        r = subprocess.run([py, os.path.join(ROOT, "tools", "fm_microbench.py"), "--json", "--ks", "19,31", "--device", str(local_rank)],
                           stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600, env=env)
        res["fm_microbench"] = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    except Exception as e:
        res["fm_microbench"] = {"error": str(e)[-200:]}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=sorted(WORKLOADS))
    ap.add_argument("--k0", type=int, default=13, help="short-prefix table length (0 = off)")
    ap.add_argument("--lanes", type=int, default=1, help="batches of one GPU in flight at once (streams + arenas); 1 with batches as large as memory allows measured best")
    ap.add_argument("--cpu-sample-mbp", type=float, default=0.0, help="Mbp of reads for the CPU baseline (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-oracle-count", action="store_true", help="skip the instrumented-oracle and issued-sector counts of the roofline (profiles/algorithmic.json is used)")
    # asked for, not default: each adds minutes after the timed steps (a FASTA file of the whole read set through the binary, twice;
    # three more workloads simulated and timed in child processes)
    ap.add_argument("--extras", action="store_true", help="add the config 2 / --nodp / index build / FM microbench sub-results")
    ap.add_argument("--cli", action="store_true", help="add the e2e_cli leg (the pbcorrect binary on a FASTA file)")
    ap.add_argument("--e2e-steps", type=int, default=2, help="timed steps of the e2e leg (after one untimed pass)")
    ap.add_argument("--batch-mbp", type=float, default=256.0, help="largest batch of reads of one lane (Mbp)")
    ap.add_argument("--nodp", action="store_true", help="disable the DP/MSA fallback on both arms (seeds + FM extension only)")
    ap.add_argument("--backend", default="nccl", choices=["nccl", "gloo"], help="process-group backend for N > 1 (gloo: tests on a one-GPU box)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed for a fixed, seeded sample of the reads as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    wl = dict(WORKLOADS[args.workload])
    if args.nodp:
        wl["desc"] += " --nodp"
    metric = "corrected Mbp/s (seed + FM-extend, --nodp)" if args.nodp else "corrected Mbp/s (seed + FM-extend + DP/MSA fallback, default options)"
    if args.impl == "reference":
        if int(os.environ.get("RANK", "0")) != 0:
            return 0
        return reference_arm(args, wl, metric)
    return ours(args, wl, metric)


if __name__ == "__main__":
    sys.exit(main())
