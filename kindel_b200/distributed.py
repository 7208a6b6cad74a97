"""Read-sharded pileup over the GPUs of one node (one process per GPU, `torch.distributed`).

The reference has no parallelism at all; SURVEY.md 8(e) defines the sharding: every record's
contribution is an independent set of +1s (reference kindel/kindel.py:40-81 has no cross-read
state) and counts are integer sums, so the coordinate-sorted read array is cut into contiguous
blocks -- one per rank -- and the only exchange step is an exact int32 sum of the seven vote
columns in front of the per-position vote (kindel.py:402-424).

Two ways to do that exchange, both bit-identical to one GPU:

  "allreduce"  NCCL all_reduce(SUM) of columns 0..6, then K2 on every rank (what the north star words).
  "peer"       the fused kernel K2p (`kdl_vote_peers_sparse`): every rank owns a slice of the slots,
               reads the seven columns of that slice straight out of the peers' tables over NVLink
               (CUDA IPC mappings), sums, votes, writes its call bytes; the call slices are then
               all-gathered (1 byte per slot).  Because the shards are blocks of sorted reads, each
               table is non-zero only on its block's footprint, and the kernel is told the
               footprints: a rank pulls just the halo (<= one read length) of its neighbours
               instead of N full tables.

Host-side helpers (`shard_batch`, `footprint`, `owner_slices`) are plain numpy and are exercised
with a 2-process gloo group on CPU in tests/test_distributed_cpu.py.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import _ffi, bamio


select_reads = bamio.select_reads


def partition_contigs(batch: bamio.ReadBatch, world: int):
    """Contigs are independent units in the reference (kindel/kindel.py:143-151): give every rank a contiguous run
    of whole contigs with about 1/world of the reads (SURVEY.md 8e, config 5: 64 contigs -> 8 per rank).  Returns
    [(c_lo, c_hi)] per rank; a rank may get nothing when there are fewer contigs than ranks."""
    cum = np.concatenate(([0], np.cumsum(np.diff(batch.contig_read_off).astype(np.int64))))
    total = int(cum[-1])
    cuts = [0]
    for r in range(1, world):
        target = total * r / world
        c = int(np.searchsorted(cum, target, side="left"))
        if c > 0 and abs(cum[c - 1] - target) <= abs(cum[min(c, len(cum) - 1)] - target):
            c -= 1
        cuts.append(min(max(c, cuts[-1]), batch.n_contigs))
    cuts.append(batch.n_contigs)
    return [(cuts[r], cuts[r + 1]) for r in range(world)]


def choose_plan(batch: bamio.ReadBatch, world: int) -> str:
    """"contigs" when there are enough contigs to give every rank whole ones of comparable weight (no slot is then
    shared between ranks: nothing to reduce), else "reads" (contiguous blocks of every contig's sorted reads)."""
    if batch.n_contigs < world:
        return "reads"
    reads = np.diff(batch.contig_read_off).astype(np.int64)
    parts = partition_contigs(batch, world)
    loads = [int(reads[a:b].sum()) for a, b in parts]
    return "contigs" if min(loads) * 2 >= max(loads) and min(loads) > 0 else "reads"


def shard_indices(batch: bamio.ReadBatch, rank: int, world: int, plan: str = "reads") -> np.ndarray:
    """Global indices of the reads rank `rank` piles (ascending)."""
    if world == 1:
        return np.arange(batch.n_reads, dtype=np.int64)
    if plan == "contigs":
        c_lo, c_hi = partition_contigs(batch, world)[rank]
        return np.arange(int(batch.contig_read_off[c_lo]), int(batch.contig_read_off[c_hi]), dtype=np.int64)
    parts = []
    for c in range(batch.n_contigs):
        lo, hi = int(batch.contig_read_off[c]), int(batch.contig_read_off[c + 1])
        parts.append(np.arange(lo + (hi - lo) * rank // world, lo + (hi - lo) * (rank + 1) // world, dtype=np.int64))
    return np.concatenate(parts) if parts else np.zeros(0, dtype=np.int64)


def shard_batch(batch: bamio.ReadBatch, rank: int, world: int) -> bamio.ReadBatch:
    """Rank's contiguous block of the reads of every contig (order and layout preserved)."""
    return batch if world == 1 else select_reads(batch, shard_indices(batch, rank, world, "reads"))


def shard_by_contig(batch: bamio.ReadBatch, rank: int, world: int) -> bamio.ReadBatch:
    """Rank's whole contigs (partition_contigs), as a batch over the SAME slot layout: its table is non-zero only
    on the slots of its own contigs, nobody else touches them, no count reduction is needed at all."""
    return select_reads(batch, shard_indices(batch, rank, world, "contigs"))


def merge_events(per_rank_events, per_rank_index) -> np.ndarray:
    """Insertion events of all shards as ONE list in the reference's iteration order: shard-local read numbers are
    mapped back to global ones, rows sorted by global read (stable: a read's own events keep their order) -- the
    rows a single GPU writes at evt_off[read] + k."""
    rows = []
    for ev, idx in zip(per_rank_events, per_rank_index):
        ev = np.asarray(ev, dtype=np.int32).reshape(-1, 4).copy()
        if ev.shape[0]:
            ev[:, 1] = np.asarray(idx, dtype=np.int64)[ev[:, 1]]
        rows.append(ev)
    allrows = np.concatenate(rows) if rows else np.zeros((0, 4), dtype=np.int32)
    return allrows[np.argsort(allrows[:, 1], kind="stable")]


def footprint(batch: bamio.ReadBatch, align: int = 4):
    """[lo, hi) slot range outside of which this shard's count table is certainly zero.
    Conservative: every read may touch from (start - its soft clips) to (start + reference span +
    clips); bounded here by SEQ length + reference-consuming CIGAR length on both sides."""
    if batch.n_reads == 0:
        return 0, 0
    per_contig = np.diff(batch.contig_read_off)
    gstart = np.repeat(batch.contig_slot, per_contig) + batch.ref_start.astype(np.int64)
    lseq = batch.seq_len.astype(np.int64)
    oplen = (batch.cigar >> 4).astype(np.int64)
    csum = np.concatenate(([0], np.cumsum(oplen)))
    span = csum[batch.cig_off[1:].astype(np.int64)] - csum[batch.cig_off[:-1].astype(np.int64)]
    reach = np.maximum(lseq, span) + 2
    lo = int((gstart - reach).min())
    hi = int((gstart + reach).max()) + 1
    # nothing a read does leaves its contig's slots [slot_c, slot_c + L_c] (a Python negative index wraps INSIDE the
    # contig's own lists, SURVEY.md A-9): the footprint lies within the contigs that have reads here
    have = np.flatnonzero(per_contig > 0)
    c_lo = int(batch.contig_slot[have[0]])
    c_hi = int(batch.contig_slot[have[-1]]) + int(batch.contig_len[have[-1]]) + 1
    # wrapping (POS == 0, or clip_starts[r_pos - 1] of a non-first S at r_pos == 0) reaches the END of the contig:
    # only KDL_HARD reads can do that, and their exact reach is not modelled here -- a shard holding a hard read that
    # starts within `reach` of its contig's start claims all of its contigs
    if batch.n_hard:
        h = batch.hard_idx.astype(np.int64)
        if (batch.ref_start[h].astype(np.int64) - reach[h] < 0).any():
            lo, hi = c_lo, c_hi
    lo, hi = max(lo, c_lo), min(hi, c_hi)
    lo = max(0, lo) // align * align
    hi = min(int(batch.n_slots), (hi + align - 1) // align * align)
    return lo, hi


def owner_slices(n_slots: int, world: int, align: int = 512):
    """Equal split of the slot space, boundaries on multiples of `align`."""
    units = n_slots // align
    cuts = [units * r // world * align for r in range(world)] + [n_slots]
    return [(cuts[r], cuts[r + 1]) for r in range(world)]


def footprint_slices(feet, n_slots: int, align: int = 64):
    """Slot ownership cut ALONG the shards' footprints: rank r votes on (roughly) the slots only its own table
    covers, the overlap with a neighbour (a halo of at most one read's reach) is cut in the middle.  Then the
    core of every slice needs no peer table at all.  Needs footprints that are ordered like the ranks (coordinate
    blocks, contig runs); anything else falls back to the equal split.  Empty shards own nothing."""
    world = len(feet)
    live = [r for r in range(world) if feet[r][1] > feet[r][0]]
    ordered = all(feet[a][0] <= feet[b][0] and feet[a][1] <= feet[b][1] for a, b in zip(live, live[1:]))
    if not ordered or not live:
        return owner_slices(n_slots, world, 512)
    bounds = [0]  # bounds[k] .. bounds[k + 1] = slice of the k-th live shard
    for a, b in zip(live, live[1:]):
        if feet[a][1] <= feet[b][0] + 4:  # disjoint (whole contigs per rank): cut exactly where b starts
            mid = feet[b][0] // 4 * 4
        else:
            mid = (feet[a][1] + feet[b][0]) // 2 // align * align
        bounds.append(min(max(mid, bounds[-1]), n_slots))
    bounds.append(n_slots)
    out, k = [], 0
    for r in range(world):
        if k < len(live) and r == live[k]:
            out.append((bounds[k], bounds[k + 1]))
            k += 1
        else:  # empty shard: zero width, where the next live slice starts
            at = bounds[k] if k < len(live) else n_slots
            out.append((at, at))
    return out


class PeerTables:
    """This rank's IPC block -- TWO count tables and TWO call buffers (epoch parity) plus the flag words -- and
    mappings of every peer's block."""

    def __init__(self, n_slots: int, device, group=None):
        import torch
        import torch.distributed as dist

        self.lib = _ffi.load()
        self.n_slots = n_slots
        self.device = device
        self.group = group
        self.world = dist.get_world_size(group)
        self.rank = dist.get_rank(group)
        # [table 0][table 1][calls 0][calls 1][flags: ready[16], done[16], counter]
        self.table_bytes = _ffi.KDL_NCOL * n_slots * 4
        self.calls_off = 2 * self.table_bytes
        self.flags_off = self.calls_off + 2 * n_slots
        nbytes = self.flags_off + 256
        ptr = C.c_void_p()
        with torch.cuda.device(device):
            _ffi.check(self.lib.kdl_table_alloc(nbytes, C.byref(ptr)), "kdl_table_alloc")
            handle = C.create_string_buffer(64)
            _ffi.check(self.lib.kdl_ipc_export(ptr, handle), "kdl_ipc_export")
        self.ptr = ptr.value
        handles = [None] * self.world
        dist.all_gather_object(handles, bytes(handle.raw), group=group)
        self.peer_ptrs = []
        self._opened = []
        with torch.cuda.device(device):
            for r, h in enumerate(handles):
                if r == self.rank:
                    self.peer_ptrs.append(self.ptr)
                    continue
                p = C.c_void_p()
                _ffi.check(self.lib.kdl_ipc_open(h, C.byref(p)), "kdl_ipc_open")
                self.peer_ptrs.append(p.value)
                self._opened.append(p.value)
        self.counts = [_wrap_device_memory(self.ptr + k * self.table_bytes, (_ffi.KDL_NCOL, n_slots), device)
                       for k in range(2)]
        self.calls = [_wrap_device_memory(self.ptr + self.calls_off + k * n_slots, (n_slots,), device, "|u1")
                      for k in range(2)]

    def exchange_struct(self, feet, slices, parity: int) -> _ffi.KdlExchange:
        x = _ffi.KdlExchange()
        x.n_ranks, x.rank = self.world, self.rank
        for r, base in enumerate(self.peer_ptrs):
            x.tables[r] = base + parity * self.table_bytes
            x.calls[r] = base + self.calls_off + parity * self.n_slots
            x.ready[r] = base + self.flags_off
            x.done[r] = base + self.flags_off + 64
            x.foot_lo[r], x.foot_hi[r] = feet[r]
            x.slice_lo[r], x.slice_hi[r] = slices[r]
        x.counter = self.ptr + self.flags_off + 128
        return x

    def close(self):
        import torch

        with torch.cuda.device(self.device):
            for p in self._opened:
                self.lib.kdl_ipc_close(p)
            self._opened = []
            if self.ptr:
                self.lib.kdl_table_free(self.ptr)
                self.ptr = None


class _CudaArray:
    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = {"shape": shape, "typestr": typestr, "data": (ptr, False), "version": 2}


def _wrap_device_memory(ptr: int, shape, device, typestr="<i4"):
    """torch view over memory this library allocated (no copy)."""
    import torch

    with torch.cuda.device(device):
        return torch.as_tensor(_CudaArray(ptr, tuple(shape), typestr), device=device)


class ShardedConsensus:
    """One rank's part of a sharded pileup + vote.  `step()` is K1 on the shard + the exchange + the vote and
    returns the COMPLETE call bytes on every rank.

    mode "fused" (default): no NCCL on the data path.  Tables and call buffers are double-buffered by epoch
    parity, so the step's only cross-rank waits are on events of the SAME step: a halo chunk of K2x waits for the
    neighbour whose footprint reaches into it (the core of a slice waits for nobody), and the gather K2g waits for
    each peer's slice.  Nothing of step n has to finish before K1 of step n+1 starts overwriting the other
    table.  "peer": the same vote kernel behind an NCCL barrier + all_gather.  "allreduce": NCCL all_reduce of
    the 7 vote columns, vote replicated (what the north star words literally; the baseline)."""

    def __init__(self, shard: bamio.ReadBatch, device, mode: str = "fused", group=None):
        import torch
        import torch.distributed as dist

        from . import engine

        self.torch, self.dist, self.engine = torch, dist, engine
        self.shard, self.device, self.mode, self.group = shard, device, mode, group
        self.world = dist.get_world_size(group)
        self.rank = dist.get_rank(group)
        self.n_slots = shard.n_slots
        self.dbatch = engine.upload(shard, device)
        self.lib = _ffi.load()
        self.epoch = 0
        if mode in ("peer", "fused"):
            self.tables = PeerTables(self.n_slots, device, group)
            feet = [None] * self.world
            dist.all_gather_object(feet, footprint(shard), group=group)
            self.feet = feet
            self.foot = feet[self.rank]
            self.slices = footprint_slices(feet, self.n_slots)
            self.xstruct = [self.tables.exchange_struct(feet, self.slices, k) for k in range(2)]
            self.foot_lo = (C.c_int64 * self.world)(*[f[0] for f in feet])
            self.foot_hi = (C.c_int64 * self.world)(*[f[1] for f in feet])
            self.ptr_arr = [(C.c_void_p * self.world)(*[p + k * self.tables.table_bytes for p in self.tables.peer_ptrs])
                            for k in range(2)]
            self.table = [engine.CountTable(self.n_slots, device, tensor=self.tables.counts[k]) for k in range(2)]
            self.sizes = [hi - lo for lo, hi in self.slices]
        elif mode == "allreduce":
            self.tables = None
            self.foot = (0, self.n_slots)
            t = torch.zeros((_ffi.KDL_NCOL, self.n_slots), dtype=torch.int32, device=device)
            self.table = [engine.CountTable(self.n_slots, device, tensor=t)] * 2
        else:
            raise ValueError("mode must be 'fused', 'peer' or 'allreduce'")
        self.counts = self.table[0].t  # (the table of the LAST step: see `last_counts`)

    @property
    def last_counts(self):
        """This rank's own count table of the most recent step (NOT reduced, except in allreduce mode)."""
        return self.table[self.epoch & 1].t

    def step(self, min_depth=1, timers=None):
        """K1 on the shard, exchange, vote.  Returns the complete call bytes on every rank.
        `timers`: optional pair of CUDA events recorded around K1 (bench.py's roofline leg)."""
        torch, dist, engine = self.torch, self.dist, self.engine
        self.epoch += 1
        par = self.epoch & 1
        table = self.table[par]
        if timers:
            timers[0].record()
        if self.mode == "allreduce":
            # the all_reduce writes sums everywhere: the whole table is dirty every step
            table.dirty = (0, self.n_slots)
            table.dirty_rest = True  # columns 5, 6 hold sums over ALL ranks after the all_reduce
            engine.pileup(self.dbatch, check=False, table=table)
        else:  # only this shard's footprint is ever touched (kdl_table_alloc zero-filled the rest)
            engine.pileup(self.dbatch, check=False, table=table, slot_range=self.foot)
        if timers:
            timers[1].record()
        if self.mode == "fused":
            st = int(torch.cuda.current_stream(self.device).cuda_stream)
            with torch.cuda.device(self.device):
                _ffi.check(self.lib.kdl_exchange_vote(C.byref(self.xstruct[par]), self.n_slots, engine.min_depth_ceil(min_depth),
                                                      self.epoch, st), "kdl_exchange_vote")
                _ffi.check(self.lib.kdl_exchange_wait(C.byref(self.xstruct[par]), self.epoch, st), "kdl_exchange_wait")
            return self.tables.calls[par]
        if self.mode == "allreduce":
            dist.all_reduce(table.t[: _ffi.KDL_NVOTE_COL], op=dist.ReduceOp.SUM, group=self.group)
            if getattr(self, "_calls_ar", None) is None:
                self._calls_ar = torch.empty(self.n_slots, dtype=torch.uint8, device=self.device)
            return engine.vote(table.t, min_depth, out=self._calls_ar)
        # "peer": every table complete before anybody reads it over NVLink
        dist.barrier(group=self.group)
        lo, hi = self.slices[self.rank]
        calls = self.tables.calls[par]
        with torch.cuda.device(self.device):
            rc = self.lib.kdl_vote_peers_sparse(
                self.ptr_arr[par], self.foot_lo, self.foot_hi, self.world, self.n_slots, lo, hi,
                engine.min_depth_ceil(min_depth), calls.data_ptr(), None,
                int(torch.cuda.current_stream(self.device).cuda_stream))
        _ffi.check(rc, "kdl_vote_peers_sparse")
        # 1 byte per slot; also the fence after which peers may overwrite this parity's tables again
        self._gather_calls(calls, lo, hi)
        return calls

    def _gather_calls(self, calls, lo, hi):
        torch, dist = self.torch, self.dist
        chunk = max(max(self.sizes), 1)
        send = torch.zeros(chunk, dtype=torch.uint8, device=self.device)
        send[: hi - lo] = calls[lo:hi]
        recv = self._recv(chunk)
        dist.all_gather_into_tensor(recv, send, group=self.group)
        for r, (a, b) in enumerate(self.slices):
            calls[a:b] = recv[r * chunk: r * chunk + (b - a)]

    def _recv(self, chunk):
        if getattr(self, "_recv_buf", None) is None or self._recv_buf.numel() != chunk * self.world:
            self._recv_buf = self.torch.empty(chunk * self.world, dtype=self.torch.uint8, device=self.device)
        return self._recv_buf

    def reduce_table(self, dst: int = 0):
        """The full 19-column table of the whole job on rank `dst` (NCCL reduce of the last step's tables; for the
        API paths that need more than call bytes: weights / features / --realign).  Returns it on `dst`, else None."""
        torch, dist = self.torch, self.dist
        t = self.last_counts.clone()
        if self.mode != "allreduce":
            dist.reduce(t, dst=dst, op=dist.ReduceOp.SUM, group=self.group)
        else:  # columns 0..6 already hold the sums everywhere; the rest still per shard
            dist.reduce(t[_ffi.KDL_NVOTE_COL:], dst=dst, op=dist.ReduceOp.SUM, group=self.group)
        return t if self.rank == dst else None

    def check_errors(self):
        """Raise the reference's exception if this rank's shard hit a data error."""
        # engine.pileup(check=False) leaves the flag unread in the hot loop; a checked pass is
        # `engine.pileup(self.dbatch)` on a scratch table, which raises exactly like one GPU.
        counts = self.torch.zeros_like(self.last_counts)
        self.engine.pileup(self.dbatch, counts, check=True)

    def close(self):
        if self.tables is not None:
            self.tables.close()
            self.tables = None


# ------------------------------------------------------------------------------------------- public entry
def _free_port() -> int:
    import socket

    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        return sk.getsockname()[1]


def _api_worker(rank: int, world: int, workdir: str, port: int, min_depth, mode: str, plan: str):
    """One process per GPU: pile this rank's shard, exchange, vote; rank 0 leaves the job's results in workdir."""
    import json
    import os
    import traceback

    import torch
    import torch.distributed as dist

    from . import engine

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", device_id=dev)
    sc = None
    try:
        batch = bamio.load_batch(os.path.join(workdir, "batch"))
        idx = shard_indices(batch, rank, world, plan)
        shard = select_reads(batch, idx)
        sc = ShardedConsensus(shard, dev, mode=mode)
        calls = sc.step(min_depth)
        # data errors: the reference raises at the FIRST offending record in iteration order -- every rank
        # reports its first one (global read number), the parent re-raises the smallest
        err = None
        try:
            sc.check_errors()
        except (IndexError, KeyError) as exc:
            read = getattr(exc, "kdl_read", None)
            err = {"type": type(exc).__name__, "args": list(exc.args),
                   "read": int(idx[read]) if read is not None and 0 <= read < idx.shape[0] else int(idx[0]) if idx.size else 0}
        errs = [None] * world
        dist.all_gather_object(errs, err)
        ev_local = sc.dbatch.tensors["_events"][: shard.n_events].cpu().numpy() if shard.n_events else np.zeros((0, 4), np.int32)
        gathered = [None] * world if rank == 0 else None
        dist.gather_object((ev_local, idx), gathered, dst=0)
        table = sc.reduce_table(0)
        if rank == 0:
            out = os.path.join(workdir, "out")
            os.makedirs(out, exist_ok=True)
            first = min((e for e in errs if e), key=lambda e: e["read"], default=None)
            with open(os.path.join(out, "status.json"), "w") as fh:
                json.dump({"error": first}, fh)
            if first is None:
                np.save(os.path.join(out, "calls.npy"), calls.cpu().numpy())
                np.save(os.path.join(out, "events.npy"), merge_events([g[0] for g in gathered], [g[1] for g in gathered]))
                np.save(os.path.join(out, "counts.npy"), table.cpu().numpy())
                np.save(os.path.join(out, "derived.npy"), engine.derive(table).cpu().numpy())
        dist.barrier()
    except Exception:  # noqa: BLE001  -- leave a trace for the parent, then fail the process
        with open(os.path.join(workdir, "rank%d.err" % rank), "w") as fh:
            fh.write(traceback.format_exc())
        raise
    finally:
        if sc is not None:
            sc.close()
        dist.destroy_process_group()


def run_sharded(batch: bamio.ReadBatch, devices: int, min_depth=1, mode: str = "fused", plan: str = None):
    """Pileup + vote of `batch` over `devices` GPUs of this node: one process per GPU (torch.distributed, NCCL for
    the plumbing, the fused peer-memory exchange on the data path), whole contigs per rank when there are enough
    of them, else contiguous blocks of every contig's sorted reads.  Returns (calls uint8[n_slots], counts
    int32[19, n_slots], derived int32[5, n_slots], events int32[n_events, 4]) in host memory -- bit-identical to
    one GPU -- or raises the reference's IndexError / KeyError."""
    import json
    import shutil
    import tempfile

    import torch
    import torch.multiprocessing as mp

    from . import engine

    engine.require_cuda()
    n_gpu = torch.cuda.device_count()
    if devices < 1 or devices > n_gpu:
        raise ValueError("devices=%d but this node has %d GPU(s)" % (devices, n_gpu))
    plan = plan or choose_plan(batch, devices)
    base = "/dev/shm" if os.path.isdir("/dev/shm") else None
    workdir = tempfile.mkdtemp(prefix="kindel_b200_", dir=base)
    try:
        bamio.save_batch(os.path.join(workdir, "batch"), batch)
        try:
            mp.spawn(_api_worker, args=(devices, workdir, _free_port(), min_depth, mode, plan), nprocs=devices, join=True)
        except Exception as exc:
            notes = []
            for r in range(devices):
                pth = os.path.join(workdir, "rank%d.err" % r)
                if os.path.exists(pth):
                    with open(pth) as fh:
                        notes.append("rank %d:\n%s" % (r, fh.read()))
            raise RuntimeError("sharded pileup failed\n" + "\n".join(notes)) from exc
        out = os.path.join(workdir, "out")
        with open(os.path.join(out, "status.json")) as fh:
            err = json.load(fh)["error"]
        if err:
            raise (KeyError if err["type"] == "KeyError" else IndexError)(*err["args"])
        return tuple(np.load(os.path.join(out, f + ".npy")) for f in ("calls", "counts", "derived", "events"))
    finally:
        shutil.rmtree(workdir, ignore_errors=True)
