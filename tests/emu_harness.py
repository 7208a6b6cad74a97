"""Builds and drives the kernel emulator (tests/emu/): test infrastructure.

`tests/emu/emu_pileup.cpp` compiles the SOURCE of K0, the tile-owner kernel K1 and every other kernel for the host on top
of `tests/emu/cuda_emu.h`, a functional model of the CUDA execution model (fibres per thread, warp
collectives, shared memory, mbarrier / bulk copy / cp.async with late completion).  `run_pileup` runs one
kernel over a batch held in numpy arrays and returns the count table."""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMU_DIR = os.path.join(ROOT, "tests", "emu")
OUT_DIR = os.path.join(EMU_DIR, "_build")
LIB = os.path.join(OUT_DIR, "libkdl_emu.so")
CUDA_INCLUDE = os.environ.get("CUDA_INCLUDE", "/usr/local/cuda/include")
F_STORE, F_ADD, F_ATOMIC = 0, 1, 2  # flush modes of the tile kernel (tile_common.cuh)

_lib = None


def available() -> bool:
    return shutil.which("g++") is not None and os.path.exists(os.path.join(CUDA_INCLUDE, "cuda_runtime.h"))


def _sources():
    csrc = os.path.join(ROOT, "kindel_b200", "csrc")
    return [os.path.join(EMU_DIR, "cuda_emu.h"), os.path.join(EMU_DIR, "emu_pileup.cpp"),
            os.path.join(csrc, "kdl_common.cuh"), os.path.join(csrc, "tile_common.cuh"), os.path.join(csrc, "pileup_tile.cu"),
            os.path.join(csrc, "pileup_general.cu"), os.path.join(csrc, "pileup_simple.cu"), os.path.join(csrc, "vote.cu"),
            os.path.join(csrc, "assemble.cu"), os.path.join(ROOT, "include", "kindel_b200.h")]


def load():
    global _lib
    if _lib is not None:
        return _lib
    src = _sources()
    if not (os.path.exists(LIB) and all(os.path.getmtime(s) <= os.path.getmtime(LIB) for s in src)):
        os.makedirs(OUT_DIR, exist_ok=True)
        cmd = ["g++", "-std=c++17", "-O1", "-g", "-fPIC", "-shared", "-I", CUDA_INCLUDE, "-I", os.path.join(ROOT, "include"),
               os.path.join(EMU_DIR, "emu_pileup.cpp"), "-o", LIB]
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError("building the kernel emulator failed:\n" + res.stdout + res.stderr)
    from kindel_b200 import _ffi

    lib = C.CDLL(LIB)
    lib.emu_last_error.restype = C.c_char_p
    lib.emu_pileup.restype = C.c_int
    lib.emu_pileup.argtypes = [C.POINTER(_ffi.KdlBatch), C.c_void_p, C.c_longlong, C.c_void_p, C.c_longlong,
                               C.c_longlong, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int]
    vp = C.c_void_p
    lib.emu_pileup_simple.argtypes = [C.POINTER(_ffi.KdlBatch), vp, C.c_longlong, vp, C.c_int]
    lib.emu_pileup_general.argtypes = [C.POINTER(_ffi.KdlBatch), vp, C.c_longlong, vp, vp, C.c_int, C.c_int]
    lib.emu_diagnose.argtypes = [C.POINTER(_ffi.KdlBatch), C.POINTER(_ffi.KdlDiag)]
    lib.emu_vote.argtypes = [vp, C.c_longlong, C.c_longlong, vp]
    lib.emu_derive.argtypes = [vp, C.c_longlong, vp]
    lib.emu_vote_peers.argtypes = [C.POINTER(vp), C.POINTER(C.c_longlong), C.POINTER(C.c_longlong), C.c_int,
                                   C.c_longlong, C.c_longlong, C.c_longlong, C.c_longlong, vp, vp]
    lib.emu_cdr_flags.argtypes = [vp, C.c_longlong, C.c_longlong, C.c_longlong, C.c_double, vp, vp]
    lib.emu_assemble.argtypes = [vp, C.c_longlong, vp, vp, C.c_int, vp, vp, vp, C.c_longlong, vp, vp, vp]
    lib.emu_set_schedule.argtypes = [C.c_int, C.c_ulonglong]
    lib.emu_set_schedule.restype = None
    lib.emu_exchange_epoch.argtypes = [C.POINTER(_ffi.KdlExchange), C.c_int, C.c_longlong, C.c_longlong, C.c_int, C.c_int]
    _lib = lib
    return lib


def _check(rc):
    if rc:
        raise RuntimeError(_lib.emu_last_error().decode())


def tileable(batch) -> bool:
    """kdl_pileup_range's test for the tile-owner path."""
    from kindel_b200 import _ffi

    return (batch.n_reads > batch.n_hard and int(batch.n_slots) % 512 == 0 and bool(batch.reads_sorted)
            and 0 < int(batch.reach_right) <= _ffi.KDL_FAST_MAXLEN + _ffi.KDL_TILE_MAXREACH)


def run_pileup(batch, mode: int = F_STORE, grid: int = 5, tile_lo: int = 0, n_tiles: int = None,
               counts: np.ndarray = None, split: int = 1, cx: bool = None, want_events: bool = False,
               zero_rest: bool = False):
    """K0 + K1 over tiles [tile_lo, tile_lo + n_tiles) of `batch` (a bamio.ReadBatch): everything but the KDL_HARD
    reads.

    mode F_STORE: the weight columns of `counts` hold garbage on entry (the kernel must overwrite them; with
    zero_rest so do columns 5..18, which the kernel zeroes in its flush before K1e adds to them);
    F_ADD / F_ATOMIC: the kernel adds to what is there (F_ATOMIC with `split` CTAs per tile).  cx: which
    instantiation (default: what kdl_pileup_range picks).  Returns int32 [19, n_slots] (and the event rows)."""
    from kindel_b200 import engine

    lib = load()
    st, keep = engine.host_struct(batch)
    n_slots = int(batch.n_slots)
    if n_tiles is None:
        n_tiles = n_slots // 512 - tile_lo
    if cx is None:
        cx = batch.n_complex > batch.n_hard
    # the table sits between two canary zones: a kernel writing outside [19, n_slots] is caught
    guard = 4096
    arena = np.full(19 * n_slots + 2 * guard, 0x7A7A7A7A, dtype=np.int32)
    table = arena[guard:guard + 19 * n_slots].reshape(19, n_slots)
    if counts is None:
        table[:] = 0
        if mode == F_STORE:
            table[0:5, tile_lo * 512:(tile_lo + n_tiles) * 512] = 0x5A5A5A5A
            if zero_rest:
                table[5:, tile_lo * 512:(tile_lo + n_tiles) * 512] = 0x3B3B3B3B
    else:
        table[:] = counts
    index = np.zeros(8 * (n_slots // 512), dtype=np.uint32)
    events = np.full((max(int(batch.n_events), 1), 4), -1, dtype=np.int32)
    rc = lib.emu_pileup(C.byref(st), table.ctypes.data, n_slots, index.ctypes.data, tile_lo, n_tiles, mode,
                        1 if cx else 0, split, events.ctypes.data, 1 if zero_rest else 0, grid)
    del keep
    if rc:
        raise RuntimeError(lib.emu_last_error().decode())
    assert (arena[:guard] == 0x7A7A7A7A).all() and (arena[-guard:] == 0x7A7A7A7A).all(), "write outside the count table"
    return (table.copy(), events[: int(batch.n_events)]) if want_events else table.copy()


def pileup_pipeline(batch, grid: int = 3, split: int = 1):
    """What kdl_pileup does, kernel by kernel, under the emulator: K0 + K1 (sorted, tileable batches) plus K1g for
    the hard reads, or K1s + K1g over every complex read (anything else); on a raised error flag, the diagnose
    kernels.  Returns (counts [19, n_slots], events [n_events, 4]) or raises IndexError / KeyError(base)
    exactly like kindel_b200.engine.pileup."""
    from kindel_b200 import _ffi, engine

    lib = load()
    st, keep = engine.host_struct(batch)
    n_slots = int(batch.n_slots)
    counts = np.zeros((19, n_slots), dtype=np.int32)
    events = np.zeros((max(int(batch.n_events), 1), 4), dtype=np.int32)
    flag = np.zeros(4, dtype=np.int32)
    if batch.n_reads:
        if tileable(batch):
            index = np.zeros(8 * (n_slots // 512), dtype=np.uint32)
            cx = batch.n_complex > batch.n_hard
            _check(lib.emu_pileup(C.byref(st), counts.ctypes.data, n_slots, index.ctypes.data, 0, n_slots // 512,
                                  F_ATOMIC if split > 1 else F_ADD, 1 if cx else 0, split, events.ctypes.data, 0, grid))
            _check(lib.emu_pileup_general(C.byref(st), counts.ctypes.data, n_slots, events.ctypes.data,
                                          flag.ctypes.data, 0, grid))
        else:
            if batch.n_reads > batch.n_complex:
                _check(lib.emu_pileup_simple(C.byref(st), counts.ctypes.data, n_slots, flag.ctypes.data, grid))
            _check(lib.emu_pileup_general(C.byref(st), counts.ctypes.data, n_slots, events.ctypes.data,
                                          flag.ctypes.data, 1, grid))
    if flag[0]:
        diag = _ffi.KdlDiag()
        _check(lib.emu_diagnose(C.byref(st), C.byref(diag)))
        assert diag.status, "error flag raised but no offending read found"
        engine.raise_like_reference(diag.status, diag.read, diag.nibble, diag.op_index)
    del keep
    return counts, events[: int(batch.n_events)]


def vote(counts: np.ndarray, min_depth=1) -> np.ndarray:
    from kindel_b200 import engine

    lib = load()
    counts = np.ascontiguousarray(counts, dtype=np.int32)
    calls = np.zeros(counts.shape[1], dtype=np.uint8)
    _check(lib.emu_vote(counts.ctypes.data, counts.shape[1], engine.min_depth_ceil(min_depth), calls.ctypes.data))
    return calls


def derive(counts: np.ndarray) -> np.ndarray:
    lib = load()
    counts = np.ascontiguousarray(counts, dtype=np.int32)
    out = np.zeros((5, counts.shape[1]), dtype=np.int32)
    _check(lib.emu_derive(counts.ctypes.data, counts.shape[1], out.ctypes.data))
    return out


def cdr_flags(counts: np.ndarray, slot_lo: int, slot_hi: int, clip_decay_threshold: float):
    """K4 over slots [slot_lo, slot_hi): (flags uint8, bases uint8) of those slots, like engine.cdr_flags."""
    lib = load()
    counts = np.ascontiguousarray(counts, dtype=np.int32)
    n_slots = counts.shape[1]
    flags = np.full(n_slots, 0xEE, dtype=np.uint8)  # (a slot the kernel skips keeps the marker)
    bases = np.full(n_slots, 0xEE, dtype=np.uint8)
    _check(lib.emu_cdr_flags(counts.ctypes.data, n_slots, int(slot_lo), int(slot_hi), float(clip_decay_threshold),
                             flags.ctypes.data, bases.ctypes.data))
    return flags[slot_lo:slot_hi].copy(), bases[slot_lo:slot_hi].copy()


def assemble(calls: np.ndarray, contig_slot, contig_len, ins_slots, ins_strings, want_offsets=False):
    """K5 over host buffers, like engine.assemble: the consensus text of every contig (list of str); with
    want_offsets also the offsets array [n_slots + 1] the scatter wrote."""
    lib = load()
    calls = np.ascontiguousarray(calls, dtype=np.uint8)
    n_slots = calls.shape[0]
    slot = np.ascontiguousarray(contig_slot, dtype=np.int64)
    length = np.ascontiguousarray(contig_len, dtype=np.int32)
    enc = [x.encode("ascii") for x in ins_strings]
    ins_off = np.zeros(len(enc) + 1, dtype=np.uint32)
    if enc:
        ins_off[1:] = np.cumsum([len(x) for x in enc])
    blob = np.frombuffer(b"".join(enc) or b"\0", dtype=np.uint8).copy()
    ins_slot = np.ascontiguousarray(ins_slots, dtype=np.int64) if enc else np.zeros(1, dtype=np.int64)
    n_blocks = (n_slots + 1 + 1023) // 1024
    sums = np.full(n_blocks + 1, 0xDEADBEEF, dtype=np.uint32)
    offsets = np.full(n_slots + 1, 0xDEADBEEF, dtype=np.uint32)
    out = np.zeros(n_slots + int(ins_off[-1]) + 16, dtype=np.uint8)
    _check(lib.emu_assemble(calls.ctypes.data, n_slots, slot.ctypes.data, length.ctypes.data, len(slot),
                            ins_slot.ctypes.data, ins_off.ctypes.data, blob.ctypes.data, len(enc), sums.ctypes.data,
                            offsets.ctypes.data, out.ctypes.data))
    starts = offsets[slot].astype(np.int64)
    ends = offsets[slot + length.astype(np.int64)].astype(np.int64)
    text = out[: int(offsets[n_slots])].tobytes()
    texts = [text[a:b].decode("ascii") for a, b in zip(starts.tolist(), ends.tolist())]
    return (texts, offsets) if want_offsets else texts


def vote_peers(tables, feet, slot_lo, slot_hi, min_depth=1, want_reduced=False):
    """K2p over host tables: vote of the SUM of `tables` on [slot_lo, slot_hi); feet = [(lo, hi)] or None."""
    from kindel_b200 import engine

    lib = load()
    n = len(tables)
    n_slots = tables[0].shape[1]
    ptrs = (C.c_void_p * n)(*[t.ctypes.data for t in tables])
    lo = (C.c_longlong * n)(*[f[0] for f in feet]) if feet else None
    hi = (C.c_longlong * n)(*[f[1] for f in feet]) if feet else None
    calls = np.zeros(n_slots, dtype=np.uint8)
    reduced = np.zeros((7, n_slots), dtype=np.int32) if want_reduced else None
    _check(lib.emu_vote_peers(ptrs, lo, hi, n, n_slots, slot_lo, slot_hi, engine.min_depth_ceil(min_depth), calls.ctypes.data,
                              reduced.ctypes.data if want_reduced else None))
    return (calls, reduced) if want_reduced else calls


def exchange_epoch(tables, feet, slices, calls, flags, epoch, min_depth=1, grid=3):
    """One epoch of the fused multi-GPU exchange (K2x on every rank, then K2g on every rank) with the ranks'
    buffers in host memory.  tables[r]: int32 [19, n_slots]; calls[r]: uint8 [n_slots]; flags: dict of per-rank
    int32 arrays 'ready', 'done' (16 each) and 'counter' (1), persistent across epochs."""
    from kindel_b200 import _ffi, engine

    lib = load()
    n = len(tables)
    n_slots = tables[0].shape[1]
    xs = (_ffi.KdlExchange * n)()
    for r in range(n):
        x = xs[r]
        x.n_ranks, x.rank = n, r
        for p in range(n):
            x.tables[p] = tables[p].ctypes.data
            x.calls[p] = calls[p].ctypes.data
            x.ready[p] = flags["ready"][p].ctypes.data
            x.done[p] = flags["done"][p].ctypes.data
            x.foot_lo[p], x.foot_hi[p] = feet[p]
            x.slice_lo[p], x.slice_hi[p] = slices[p]
        x.counter = flags["counter"][r].ctypes.data
    _check(lib.emu_exchange_epoch(xs, n, n_slots, engine.min_depth_ceil(min_depth), epoch, grid))


def set_schedule(mode: str = "forward", seed: int = 1):
    """Order in which the emulator runs the threads of a block within a scheduler round: "forward", "reverse" or
    "random" (a fresh pseudo-random order every round) -- different interleavings of producers and consumers."""
    load().emu_set_schedule({"forward": 0, "reverse": 1, "random": 2}[mode], seed)
