#!/usr/bin/env python
"""bench.py -- aligned bases / second through pileup + consensus (BASELINE.json's metric).

    python bench.py --gpus 1 --warmup 5                        # this engine, 1 GPU, >= 0.5 s of timed steps
    torchrun ... bench.py --gpus N ...                         # sharded over N GPUs (one process per GPU)
    python bench.py --impl reference ...                       # the reference's own CPU functions, same metric

A "step" is one pass of the hot path over one batch: K0 tile index + K1 pileup over every read (into a reused
table: nothing is memset), (N > 1: the count exchange across ranks), K2 vote over every position.

Workload (config.workload), default `cfg4_5Mb_200x` = BASELINE.json configs[3] as SURVEY.md 8(d) specifies it:
synthetic 5 Mb contig, 200x, 150 bp reads, coordinate-sorted, "mostly 150M with ~1 % indel/clip reads", 1 %
substitutions (6.67 M reads, ~10^9 aligned bases).  For N > 1 every rank gets that full per-GPU workload on its own
1/N slice of the coordinate range (weak scaling: a coordinate-sorted, N x deeper alignment cut into N contiguous
read blocks); the fixed 5 Mb x 200x set cut N ways (strong scaling) is measured in the same run and reported
beside it (`strong_scaling`).  `cfg5_64x100kb_500x` is partitioned by contig (8 contigs per rank at N = 8: no
slot is shared, nothing is reduced).  Other workloads: --workload (cfg2, cfg3, cfg5, all-simple cfg4, 30 % complex).

Numbers on the JSON line:
  value         whole-job aligned bases/s with the flattened reads already resident in HBM; CUDA events on the
                launch stream, max over ranks, over exactly --steps back-to-back steps or, without --steps, as
                many as cover >= 0.5 s of device time (`steps_timed`; `steps` echoes the request);
                `step_ms` = min / median / p90 / max of the individual steps.
  e2e           the same metric from HOST buffers, mean over max(3, min(steps_timed, 10)) calls: N = 1 through the C-ABI call kdl_ctx_consensus (pinned host
                buffers in, H2D + kernels + D2H of the call bytes inside the timed region); N > 1 through the whole
                sharded job (every rank's H2D of its shard + K1 + exchange + vote + D2H of the complete call bytes).
  roofline      dominant kernel (K0 + K1) against the measured HBM copy bandwidth (MEASURED_PEAKS.json).
  parity        sha256 of the call bytes the timed loop produced == sha256 of the CPU oracle's calls for the same job.
  cpu_baseline  the reference's own functions on this box's host CPU, bounded sample (see --impl reference).
Inputs are larger than L2 (126 MB) for the cfg4 / cfg5 workloads (no flush needed); the small ones (cfg2, cfg3)
fit in L2 and say so in config.l2_policy.

--dump-outputs DIR writes what the last timed step computed -- the count table, the insertion-event rows and the
call bytes a caller of pileup + vote receives (N > 1: the call bytes) -- as DIR/<name>.npy in float32 (float64
where float32 would round), at most DUMP_BYTES in all: an array that does not fit keeps a fixed, seeded sample of
its slots / rows, and DIR/<name>_index.npy says which.  The workloads are generated from fixed seeds, so two builds
run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "aligned bases/sec through pileup+consensus"
UNIT = "aligned_bases/s"
MIN_TIMED_S = 0.5  # without --steps, the headline rests on at least this much device time
DUMP_BYTES = 60_000_000  # --dump-outputs: the data of all arrays together (each .npy adds a 128-byte header)

WORKLOADS = {
    # name: (contig lengths, depth, fraction of indel/clip reads or "cfg3", N > 1 partition)
    "cfg4_5Mb_200x": ([5_000_000], 200, 0.01, "reads"),
    "cfg4_5Mb_200x_simple": ([5_000_000], 200, 0.0, "reads"),
    "cfg4_5Mb_200x_30pct_complex": ([5_000_000], 200, 0.30, "reads"),
    "cfg2_30kb_2000x": ([30_000], 2000, 0.0, "reads"),
    "cfg3_30kb_5000x": ([30_000], 5000, "cfg3", "reads"),
    "cfg5_64x100kb_500x": ([100_000] * 64, 500, 0.0, "contigs"),
    "tiny": ([200_000], 50, 0.05, "reads"),
}


def gen_reads(name, start_frac=None, read_seed=None):
    from kindel_b200 import synth

    lens, depth, cx, _ = WORKLOADS[name]
    if cx == "cfg3":
        return synth.complex_reads(3, lens[0], depth, start_frac=start_frac, read_seed=read_seed,
                                   edge_tail=start_frac is None)
    if cx:
        return synth.mixed_reads(4, lens, depth, cx, start_frac=start_frac, read_seed=read_seed)
    return synth.simple_reads(4, lens, depth, start_frac=start_frac, read_seed=read_seed)


def make_workload(name, rank=0, world=1, scaling="weak"):
    """(this rank's reads, the whole job's aligned bases or None = sum over the ranks, how the job is cut).

    weak   (default): every rank gets the full per-GPU workload -- `depth` x the contig lengths worth of
           reads -- placed on its own 1/N slice of the coordinate range (a coordinate-sorted N x deeper
           BAM cut into N contiguous blocks): per-GPU work is fixed as N grows.
    strong: the N = 1 data set cut N ways: contiguous read blocks, or whole contigs for the multi-contig workload."""
    from kindel_b200 import bamio, distributed

    part = WORKLOADS[name][3]
    if world == 1:
        full = gen_reads(name)
        return full, full.aligned_bases, "none"
    if part == "contigs":  # config 5: contigs are independent units -> whole contigs per rank, no reduction at all
        full = gen_reads(name)
        if scaling == "strong":
            return distributed.shard_by_contig(full, rank, world), full.aligned_bases, "whole contigs per rank"
        # weak: N x the contigs (N x 64 x 100 kb), each rank its own 64 -- the same per-GPU work as N = 1
        lens = WORKLOADS[name][0]
        all_lens = lens * world
        names = ["ctg%d" % i for i in range(len(all_lens))]
        read_off = np.zeros(len(all_lens) + 1, dtype=np.int64)
        k0 = rank * len(lens)
        read_off[k0 + 1:k0 + len(lens) + 1] = full.contig_read_off[1:]
        read_off[k0 + len(lens) + 1:] = full.n_reads
        shard = bamio.finalize(names, np.asarray(all_lens), read_off, full.ref_start, full.seq_off, full.seq_len,
                               full.cig_off, full.cigar, full.seq4, n_records=full.n_reads)
        return shard, full.aligned_bases * world, "whole contigs per rank (N x the contigs)"
    if scaling == "strong":
        full = gen_reads(name)
        return distributed.shard_batch(full, rank, world), full.aligned_bases, "contiguous blocks of the sorted reads"
    shard = gen_reads(name, start_frac=(rank / world, (rank + 1) / world), read_seed=[4, rank])
    return shard, None, "contiguous blocks of the sorted reads (N x deeper in total)"


def algorithmic_bytes(batch):
    """SURVEY.md 8(d): per read ceil(l_seq/2) + 4*n_cigar + 12 read-side bytes (K1);
    per position 28 B read + 1 B written by the vote (K2)."""
    lseq = batch.seq_len.astype(np.int64)
    n_cig = np.diff(batch.cig_off.astype(np.int64))
    k1 = int(((lseq + 1) // 2).sum() + 4 * n_cig.sum() + 12 * batch.n_reads)
    k2 = int(batch.n_slots) * 29
    return k1, k2


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region.  Started well before it: the tool's
    own start-up (NVML initialisation over every GPU of the box) must not land inside the timed steps."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []
        self.t_mark = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def wait_first_sample(self, timeout=10.0):
        t0 = time.time()
        while self.proc and not self.lines and time.time() - t0 < timeout:
            time.sleep(0.05)

    def mark(self):
        """Samples from here on count (the timed region starts)."""
        self.t_mark = len(self.lines)

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.lines[(self.t_mark or 0):]:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for k, nm in enumerate(names):
                if f[5 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(workload, world):
    """dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel, per launch, from the committed
    `ncu --set full` capture of this same command (profiles/); None for configurations not captured."""
    if world != 1:
        return None
    try:
        with open(os.path.join(ROOT, "profiles", "r02_k1_traffic.json")) as fh:
            d = json.load(fh).get(workload)
        return int(d["dram_bytes_read"]) + int(d["dram_bytes_write"]) if d else None
    except Exception:
        return None


def quantiles(xs):
    xs = sorted(xs)
    n = len(xs)
    return {"min": xs[0], "median": xs[n // 2], "p90": xs[min(n - 1, int(0.9 * n))], "max": xs[-1]}


# ------------------------------------------------------------------------------ CPU baselines
def cpu_sample_records(batch, target_bases=5.0e7):
    """Record objects of a bounded window of the workload: the first reads of contig 0 (about `target_bases`
    aligned bases) against a contig truncated behind the last of them."""
    from oracle import py_oracle

    L0 = int(batch.contig_len[0])
    n0 = int(batch.contig_read_off[1])
    per_read = max(1.0, batch.aligned_bases / max(1, batch.n_reads))
    want_reads = max(1, int(target_bases / per_read))
    if want_reads >= n0:
        hi, window = n0, L0
    else:
        hi = want_reads
        reach = int(max(batch.reach_right, int(batch.seq_len[:hi].max()))) + 64
        window = min(L0, int(batch.ref_start[:hi].max()) + reach)
    recs = py_oracle.records_of(batch, 0, hi)
    bases = sum(n for r in recs for n, op in r.cigars if op in ("M", "=", "X"))
    return recs, bases, window


def load_cpu_reference():
    """(module or None, kind, description): the unmodified reference if a tree is found, else the port."""
    kind, how = "port", "oracle/py_oracle.py (reference-shaped CPython port; no reference tree found)"
    ref = None
    try:
        from oracle import refload

        if refload.available():
            ref = refload.load_reference()
            kind = "reference"
            how = ("unmodified reference kindel/kindel.py (%s): parse_records + consensus_sequence"
                   % os.path.relpath(refload.REFERENCE_ROOT, ROOT))
    except Exception as exc:  # noqa: BLE001
        how += " (loading the reference failed: %s)" % exc
        ref = None
    return ref, kind, how


def cpu_reference_pass(ref, recs, window):
    """One pass of the reference's hot path over the sample; seconds."""
    t0 = time.perf_counter()
    if ref is not None:
        aln = ref.parse_records("ctg0", window, recs)
        ref.consensus_sequence(aln.weights, aln.insertions, aln.deletions, None, False, 1, False)
    else:
        from oracle import py_oracle

        p = py_oracle.pileup(window, recs)
        py_oracle.vote(p, 1)
    return time.perf_counter() - t0


def cpu_reference_sample(batch, target_bases=5.0e7):
    """The reference's OWN functions (unmodified kindel/kindel.py, staged under oracle/_ref by
    oracle/stage_reference.py; loaded through oracle/refload.py's import stubs): parse_records +
    consensus_sequence (kindel.py:21-128, 384-430) on a bounded sample, single core -- the reference has no
    parallelism (kindel/kindel.py:1-14 imports no threading / multiprocessing).  Falls back to the
    reference-shaped CPython port (oracle/py_oracle.py) when no reference tree can be found; says which ran."""
    recs, bases, window = cpu_sample_records(batch, target_bases)
    ref, kind, how = load_cpu_reference()
    dt = cpu_reference_pass(ref, recs, window)
    return {"value": bases / dt, "unit": UNIT, "cores": 1, "kind": kind,
            "sample": "%s; %d reads / %d aligned bases over the first %d positions of the workload, %.1f s"
                      % (how, len(recs), bases, window, dt)}


def cpu_native_sample(batch):
    """The C restatement (oracle/kindel_oracle.c), 1 thread, whole shard: what a compiled CPU loop does."""
    from oracle import coracle

    t0 = time.perf_counter()
    counts, _ = coracle.pileup(batch)
    coracle.vote(counts, 1)
    dt = time.perf_counter() - t0
    return {"value": batch.aligned_bases / dt, "unit": UNIT, "cores": 1, "kind": "port-native",
            "sample": "oracle/kindel_oracle.c single thread, full workload, %.2f s" % dt}


def host_side_timings(batch):
    """The host work that surrounds the timed spans (SURVEY.md 8d: reported separately; it stays on the host in
    both paths): decode of a real BGZF-compressed BAM of 10^6 reads of the workload's shape (150 bp, coordinate-sorted)
    by the C++ decoder -- inflate, filter, classification, device layout -- on this box's cores."""
    import tempfile

    from kindel_b200 import bamio, synth

    sub = synth.simple_reads(4, [750_000], 200)  # 10^6 reads, 1.5e8 aligned bases
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "slice.bam")
        synth.write_simple_bam(path, sub)
        size = os.path.getsize(path)
        best = None
        for _ in range(3):
            t0 = time.perf_counter()
            back = bamio.read_bam(path)
            dt = time.perf_counter() - t0
            best = dt if best is None or dt < best else best
        # the whole user-visible job on that file: decode + H2D + K0..K2 + K5 + D2H + FASTA records
        from kindel_b200 import kindel as K

        wall = None
        for _ in range(2):
            t0 = time.perf_counter()
            res = K.bam_to_consensus(path)
            dt = time.perf_counter() - t0
            wall = dt if wall is None or dt < wall else wall
        fasta_bases = sum(len(c.sequence) for c in res.consensuses)
    assert back.n_reads == sub.n_reads and np.array_equal(back.seq4, sub.seq4)
    return {"file_to_fasta_wall_s": wall, "file_to_fasta_aligned_bases_per_s": back.aligned_bases / wall,
            "file_to_fasta_note": "kindel.bam_to_consensus(path) on the same file: %d consensus bases (best of 2)" % fasta_bases,
            "bam_decode_flatten_reads_per_s": sub.n_reads / best,
            "bam_decode_flatten_aligned_bases_per_s": back.aligned_bases / best,
            "sample": "%d reads, %.0f MB BGZF BAM, C++ decoder (kdl_bam_*: inflate + filter + classify + fill, %d threads): "
                      "%.3f s (best of 3)" % (sub.n_reads, size / 1e6, bamio.decode_threads(), best),
            "cores": os.cpu_count()}


def run_reference(args):
    """`--impl reference`: W untimed + K timed passes of the reference's own parse_records + consensus_sequence over
    a bounded sample of the workload, one host core (the reference has no parallelism).  The sample is sized so that
    the K + W passes take about 2 minutes in all (at most 5e7 aligned bases, ~6 s, per pass)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    batch, total, _ = make_workload(args.workload)
    passes = max(1, args.steps) + max(0, args.warmup)
    target = min(5.0e7, max(2.0e6, 8.0e6 * 120.0 / passes))  # ~8e6 bases/s for the reference on this class of host
    recs, bases, window = cpu_sample_records(batch, target)
    ref, kind, how = load_cpu_reference()
    for _ in range(max(0, args.warmup)):
        cpu_reference_pass(ref, recs, window)
    times = [cpu_reference_pass(ref, recs, window) for _ in range(max(1, args.steps))]
    dt = statistics.median(times)
    v = bases / dt
    native = cpu_native_sample(batch)
    cpu = {"value": v, "unit": UNIT, "cores": 1, "kind": kind,
           "sample": "%s; %d reads / %d aligned bases over the first %d positions of the workload per step, median of "
                     "%d steps %.2f s (min %.2f, max %.2f)" % (how, len(recs), bases, window, len(times), dt, min(times), max(times))}
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "int32", "data": "synthetic",
        "config": {"workload": args.workload, "note": "reference is single-threaded CPython (kindel/kindel.py:1-14); "
                   "a step = one pass over a bounded sample of the workload"},
        "cpu_baseline": cpu,
        "cpu_native_port": native,
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "host": {"nproc": os.cpu_count()},
    }
    print(json.dumps(line))
    return 0


# ----------------------------------------------------------------------------------- GPU arm
def time_steps(step, steps, warmup, torch, dist, world, dev, min_seconds=MIN_TIMED_S):
    """W warm-up steps, then exactly `steps` back-to-back steps -- or, if `steps` is None, as many as cover
    >= min_seconds of device time at the step time of 3 more untimed steps; one CUDA event triple per step
    (dispersion, K1 / K2 split) -- the region is bracketed by the first and last events."""
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    if steps is not None:
        reps = max(1, steps)
    else:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(3):
            step()
        e1.record()
        torch.cuda.synchronize()
        est_ms = max(e0.elapsed_time(e1) / 3, 1e-3)
        reps = min(int(math.ceil(min_seconds * 1e3 / est_ms)), 20000)
        if world > 1:  # every rank must run the same number of steps
            t = torch.tensor([reps], dtype=torch.int64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            reps = int(t.item())
    if world > 1:
        dist.barrier()
    ev = [tuple(torch.cuda.Event(enable_timing=True) for _ in range(3)) for _ in range(reps)]
    ev_end = torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    out = None
    for i in range(reps):
        out = step(ev[i])
    ev_end.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    total_ms = ev[0][0].elapsed_time(ev_end)
    step_ms = [ev[i][0].elapsed_time(ev[i + 1][0]) for i in range(reps - 1)] + [ev[-1][0].elapsed_time(ev_end)]
    k1_ms = [e[0].elapsed_time(e[1]) for e in ev]
    k2_ms = [e[1].elapsed_time(e[2]) for e in ev]
    return {"reps": reps, "total_ms": total_ms, "step_ms": step_ms, "k1_ms": statistics.mean(k1_ms),
            "k2_ms": statistics.mean(k2_ms), "out": out}


def dump_outputs(out_dir, arrays, budget=DUMP_BYTES):
    """arrays: {name: (numpy array, axis along which it may be sampled)} -> out_dir/<name>.npy.  Smaller arrays are
    written whole; the budget left is shared among the larger ones, which keep a seeded sample along their axis."""
    os.makedirs(out_dir, exist_ok=True)
    items = sorted(arrays.items(), key=lambda kv: kv[1][0].size)
    left = budget
    for i, (name, (a, axis)) in enumerate(items):
        a = np.asarray(a)
        dt = np.float32 if a.size == 0 or np.abs(a).max() < 2 ** 24 else np.float64
        share = left // (len(items) - i)
        n = a.shape[axis]
        per = np.dtype(dt).itemsize * (a.size // max(n, 1))
        if per * n > share:
            k = max(1, share // (per + 8))  # + the float64 index of each kept slot / row
            idx = np.sort(np.random.default_rng(0).choice(n, size=k, replace=False))
            a = np.take(a, idx, axis=axis)
            np.save(os.path.join(out_dir, name + "_index.npy"), idx.astype(np.float64))
            left -= 8 * k
        out = np.ascontiguousarray(a, dtype=dt)
        np.save(os.path.join(out_dir, name + ".npy"), out)
        left -= out.nbytes


def oracle_digest(batch, torch, dist, world, dev, min_depth=1):
    """sha256 of the CPU oracle's call bytes for the whole job: every rank piles ITS shard with the C oracle, the
    7 vote columns are summed across ranks (an integer all_reduce: plumbing), the oracle votes."""
    from oracle import coracle

    counts, _ = coracle.pileup(batch)
    if world > 1:
        t = torch.from_numpy(np.ascontiguousarray(counts[:7])).to(dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        counts = np.zeros_like(counts)
        counts[:7] = t.cpu().numpy()
    calls = coracle.vote(counts, min_depth)
    return hashlib.sha256(calls.tobytes()).hexdigest()


def run_native(args):
    import torch
    import torch.distributed as dist

    from kindel_b200 import _ffi, engine

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit("--gpus must equal WORLD_SIZE under torchrun")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _ffi.load()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()  # long before the timed region: its start-up must not stall any launch inside it

    def build_case(scaling):
        batch, total, sharding = make_workload(args.workload, rank, world, scaling)
        if total is None:
            t = torch.tensor([batch.aligned_bases], dtype=torch.int64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            total = int(t.item())
        if world == 1:
            db = engine.upload(batch, dev)
            table = engine.CountTable(batch.n_slots, dev)
            calls_buf = torch.empty(batch.n_slots, dtype=torch.uint8, device=dev)

            def step(timers=None):
                # a fresh pileup into a reused table: nothing is memset, K1 overwrites the weight columns
                if timers:
                    timers[0].record()
                counts, events = engine.pileup(db, check=False, table=table)
                if timers:
                    timers[1].record()
                calls = engine.vote(table.t, 1, out=calls_buf)
                if timers:
                    timers[2].record()
                return {"counts": counts, "events": events, "calls": calls}
            return batch, total, sharding, step, None
        from kindel_b200 import distributed

        sc = distributed.ShardedConsensus(batch, dev, mode=args.exchange)

        def step(timers=None):
            calls = sc.step(1, timers)
            if timers:
                timers[2].record()
            return {"calls": calls}
        return batch, total, sharding, step, sc

    batch, total_bases, sharding, step, sc = build_case(args.scaling)
    n_slots = batch.n_slots
    k1_bytes, k2_bytes = algorithmic_bytes(batch)
    if rank == 0:
        sampler.wait_first_sample()
    launches0 = lib.kdl_launch_count()
    if rank == 0:
        sampler.mark()
    tm = time_steps(step, args.steps, args.warmup, torch, dist, world, dev)
    launches = lib.kdl_launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    launches_per_step = launches / (args.warmup + (0 if args.steps is not None else 3) + tm["reps"])
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {name: (t.cpu().numpy(), 1 if name == "counts" else 0)
                                         for name, t in tm["out"].items()})
    # parity of what the timed loop produced (outside the timed region)
    got = hashlib.sha256(tm["out"]["calls"].cpu().numpy().tobytes()).hexdigest()
    want = oracle_digest(batch, torch, dist, world, dev)
    t = torch.tensor([tm["total_ms"], tm["k1_ms"], tm["k2_ms"], 0.0 if got == want else 1.0], dtype=torch.float64,
                     device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, k1_ms_max, k2_ms_max, parity = float(t[0]), float(t[1]), float(t[2]), float(t[3]) == 0.0
    ms_per_step = total_ms / tm["reps"]
    value = total_bases / (ms_per_step * 1e-3)
    step_q = quantiles(tm["step_ms"])

    # ---- e2e from pinned HOST buffers ---------------------------------------------------------------
    n_e2e = max(3, min(tm["reps"], 10))
    if world == 1:
        ctx = engine.HostContext(local)
        pinned = {}
        for f in engine._FIELDS:
            a = np.ascontiguousarray(getattr(batch, f))
            pinned[f] = torch.from_numpy(a.view(np.int32) if a.dtype == np.uint32 else a).pin_memory() if a.size else None
        ptr = {f: (int(tp.data_ptr()) if tp is not None else None) for f, tp in pinned.items()}
        struct = engine.make_struct(batch, ptr)
        calls_host = torch.empty(n_slots, dtype=torch.uint8).pin_memory()
        calls_np = calls_host.numpy()
        rows = []
        for i in range(2 + n_e2e):
            t0 = time.perf_counter()
            ctx.consensus(batch, 1, calls_out=calls_np, struct=struct)
            wall = (time.perf_counter() - t0) * 1e3
            tmg = ctx.last_timing()
            rows.append((tmg["h2d_ms"] + tmg["kernel_ms"] + tmg["d2h_ms"], wall, tmg))
        rows = rows[-n_e2e:]
        dev_ms = statistics.mean(x[0] for x in rows)
        e2e = {"value": total_bases / (dev_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": batch.input_bytes(),
               "d2h_bytes_per_step": int(n_slots) + 16, "ms_per_step": dev_ms,
               "wall_ms_per_step": statistics.mean(x[1] for x in rows),
               "breakdown_ms": {k: statistics.mean(x[2][k] for x in rows) for k in ("h2d_ms", "kernel_ms", "d2h_ms")},
               "parity": hashlib.sha256(calls_np.tobytes()).hexdigest() == want,
               "api": "kdl_ctx_consensus (include/kindel_b200.h), pinned host buffers"}
        ctx.close()
    else:
        # the whole sharded job from host memory: every rank copies its shard in, piles, exchanges, votes, and
        # copies the COMPLETE call bytes out (rank 0's copy is the job's result; every rank does it, symmetric)
        dbt = sc.dbatch.tensors
        pinned = {f: dbt[f].cpu().pin_memory() for f in engine._FIELDS}
        calls_host = torch.empty(n_slots, dtype=torch.uint8).pin_memory()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        times = []
        for i in range(2 + n_e2e):
            dist.barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ev[0].record()
            for f in engine._FIELDS:
                dbt[f].copy_(pinned[f], non_blocking=True)
            calls = sc.step(1)
            calls_host.copy_(calls, non_blocking=True)
            ev[1].record()
            torch.cuda.synchronize()
            times.append((ev[0].elapsed_time(ev[1]), (time.perf_counter() - t0) * 1e3))
        times = times[-n_e2e:]
        e2e_ok = hashlib.sha256(calls_host.numpy().tobytes()).hexdigest() == oracle_digest(batch, torch, dist, world, dev)
        tt = torch.tensor([statistics.mean(x[0] for x in times), statistics.mean(x[1] for x in times),
                           0.0 if e2e_ok else 1.0], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e = {"value": total_bases / (float(tt[0]) * 1e-3), "unit": UNIT,
               "h2d_bytes_per_step": int(sum(pinned[f].numel() * pinned[f].element_size() for f in engine._FIELDS)),
               "d2h_bytes_per_step": int(n_slots), "ms_per_step": float(tt[0]), "wall_ms_per_step": float(tt[1]),
               "parity": float(tt[2]) == 0.0,
               "api": "distributed.ShardedConsensus.step from pinned host buffers: per rank H2D of its shard, K0 + K1, "
                      "exchange + vote, D2H of the complete call bytes (byte counts are per rank; time = max over ranks)"}

    # ---- strong scaling beside the weak line (N > 1): the fixed N = 1 data set cut N ways
    strong = None
    if world > 1 and args.scaling == "weak" and not args.no_strong:
        sb, s_total, s_sharding, s_step, s_sc = build_case("strong")
        stm = time_steps(s_step, args.steps, args.warmup, torch, dist, world, dev, min_seconds=0.25)
        s_got = hashlib.sha256(stm["out"]["calls"].cpu().numpy().tobytes()).hexdigest()
        s_par = s_got == oracle_digest(sb, torch, dist, world, dev)
        tt = torch.tensor([stm["total_ms"], stm["k1_ms"], 0.0 if s_par else 1.0], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        s_ms = float(tt[0]) / stm["reps"]
        strong = {"scaling": "strong", "workload": args.workload, "sharding": s_sharding,
                  "aligned_bases_total": int(s_total), "ms_per_step": s_ms, "value": s_total / (s_ms * 1e-3),
                  "unit": UNIT, "steps_timed": stm["reps"], "step_ms": quantiles(stm["step_ms"]),
                  "k0_k1_ms": float(tt[1]), "parity": float(tt[2]) == 0.0}
        s_sc.close()
        del sb, s_step, s_sc

    if rank == 0:
        peak, peak_src = measured_peak()
        achieved = k1_bytes / (k1_ms_max * 1e-3) / 1e9
        in_mb = batch.input_bytes() / 1e6
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "int32", "data": "synthetic",
            "steps_timed": tm["reps"], "timed_region_s": total_ms * 1e-3, "step_ms": step_q,
            "parity": parity,
            "config": {"workload": args.workload if world == 1 or args.scaling == "strong" else
                       "%s per GPU (%dx in total)" % (args.workload, world),
                       "reads_per_rank": int(batch.n_reads), "complex_reads_per_rank": int(batch.n_complex),
                       "aligned_bases_total": int(total_bases),
                       "sharding": sharding,
                       "reduction": ("none" if world == 1 else
                                     "K2x/K2g: flags + footprint-clipped reduce + vote + call gather over CUDA-IPC peer "
                                     "memory (NVLink), tables double-buffered by epoch; no NCCL on the data path"
                                     if args.exchange == "fused" else
                                     "K2p: vote over peer tables (NVLink), NCCL barrier + all_gather of call bytes"
                                     if args.exchange == "peer" else
                                     "NCCL all_reduce(int32 sum) of the 7 vote columns, vote replicated"),
                       "l2_policy": ("inputs (%.0f MB) larger than L2 (126 MB); no flush" % in_mb if in_mb > 126 else
                                     "inputs (%.0f MB) fit in L2 (126 MB) and stay there between steps: a small-reference "
                                     "workload, reported as it runs" % in_mb)},
            "roofline": {"bound": "hbm", "kernel": "K0 tile index + K1 tile-owner pileup",
                         "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak, "traffic": ncu_traffic(args.workload, world),
                         "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": k1_bytes, "kernel_ms": k1_ms_max},
            "kernels_ms": {"k0_k1_pileup": k1_ms_max, "k2_vote_or_exchange": k2_ms_max,
                           "k2_vote_gbs": (k2_bytes / (k2_ms_max * 1e-3) / 1e9) if world == 1 and k2_ms_max else None},
            "e2e": e2e, "gpu_launches": int(round(launches_per_step * tm["reps"])),
            "gpu_launches_per_step": launches_per_step, "clocks": clocks,
        }
        if strong is not None:
            line["strong_scaling"] = strong
        if world == 1 and not args.no_cpu:
            line["cpu_baseline"] = cpu_reference_sample(batch)
            line["cpu_native_port"] = cpu_native_sample(batch)
            line["host"] = host_side_timings(batch)
        print(json.dumps(line))
    if sc is not None:
        sc.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps, exactly (default: as many as cover >= 0.5 s of device time; --impl reference: 20)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", choices=["native", "reference"], default="native")
    ap.add_argument("--workload", choices=sorted(WORKLOADS), default="cfg4_5Mb_200x")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (float32/float64, seeded sample "
                         "of arrays beyond the size budget)")
    ap.add_argument("--no-strong", action="store_true", help="N > 1: skip the strong-scaling measurement beside the weak one")
    ap.add_argument("--scaling", choices=["weak", "strong"], default="weak",
                    help="N > 1: weak = the full per-GPU workload on every rank (N x deeper in total); "
                         "strong = the N = 1 data set cut N ways")
    ap.add_argument("--exchange", choices=["fused", "peer", "allreduce"], default="fused",
                    help="N > 1: fused = flags + reduce + vote + call gather over NVLink peer memory (no NCCL on "
                         "the data path); peer = same vote kernel with NCCL barrier/all_gather; allreduce = NCCL "
                         "all_reduce of the vote columns, vote replicated")
    args = ap.parse_args()
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        if args.steps is None:
            args.steps = 20
        return run_reference(args)
    return run_native(args)


if __name__ == "__main__":
    raise SystemExit(main())
