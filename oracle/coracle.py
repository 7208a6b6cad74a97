"""TEST INFRASTRUCTURE ONLY -- ctypes front-end of oracle/kindel_oracle.c (the CPU checker).

Takes any object exposing the flattened-batch attributes of include/kindel_b200.h as numpy arrays
(duck-typed; this module does not import the product package) and returns plain numpy results:

    pileup(batch)  -> (counts int32[19, n_slots], events int32[n_events, 4])   or raises
                      IndexError / KeyError exactly where the reference would (SURVEY.md A-10)
    vote(counts, min_depth) -> calls uint8[n_slots]
    derive(counts) -> int32[5, n_slots]

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may use it.
"""
from __future__ import annotations

import ctypes as C
import math
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "kindel_oracle.c")
_LIB = os.path.join(_HERE, "_build", "libkindel_oracle.so")
NIBBLES = "=ACMGRSVTWYHKDBN"
NCOL = 19


class _Batch(C.Structure):
    _fields_ = [
        ("n_reads", C.c_int64), ("n_ops", C.c_int64), ("seq4_words", C.c_int64),
        ("ref_start", C.c_void_p), ("seq_off", C.c_void_p), ("l_seq", C.c_void_p),
        ("cig_off", C.c_void_p), ("cigar", C.c_void_p), ("seq4", C.c_void_p),
        ("n_contigs", C.c_int32), ("reads_sorted", C.c_int32), ("max_simple_len", C.c_int32), ("reserved0", C.c_int32),
        ("contig_read_off", C.c_void_p), ("contig_len", C.c_void_p), ("contig_slot", C.c_void_p),
        ("n_complex", C.c_int64), ("complex_idx", C.c_void_p), ("evt_off", C.c_void_p),
    ]


class _Diag(C.Structure):
    _fields_ = [("status", C.c_int32), ("reserved", C.c_int32), ("read", C.c_int64),
                ("nibble", C.c_int32), ("op_index", C.c_int32)]


_lib = None


def build(force: bool = False) -> str:
    if force or not os.path.exists(_LIB) or os.path.getmtime(_LIB) < os.path.getmtime(_SRC):
        os.makedirs(os.path.dirname(_LIB), exist_ok=True)
        subprocess.run(["gcc", "-O2", "-fPIC", "-shared", "-std=c11", "-Wall", _SRC, "-o", _LIB], check=True)
    return _LIB


def _load():
    global _lib
    if _lib is None:
        lib = C.CDLL(build())
        lib.oracle_pileup.restype = C.c_int
        lib.oracle_pileup.argtypes = [C.POINTER(_Batch), C.c_void_p, C.c_int64, C.c_void_p,
                                      C.POINTER(C.c_int64), C.POINTER(_Diag)]
        lib.oracle_vote.restype = None
        lib.oracle_vote.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p]
        lib.oracle_derive.restype = None
        lib.oracle_derive.argtypes = [C.c_void_p, C.c_int64, C.c_void_p]
        _lib = lib
    return _lib


def _struct(batch, keep):
    def ptr(a, dtype):
        a = np.ascontiguousarray(a, dtype=dtype)
        keep.append(a)
        return a.ctypes.data

    b = _Batch()
    b.n_reads = int(batch.ref_start.shape[0])
    b.n_ops = int(batch.cigar.shape[0])
    b.seq4_words = int(batch.seq4.shape[0])
    b.ref_start = ptr(batch.ref_start, np.int32)
    b.seq_off = ptr(batch.seq_off, np.uint32)
    # plain SEQ lengths: the checker does not depend on the device word's flag bits
    b.l_seq = ptr(batch.seq_len if getattr(batch, "seq_len", None) is not None else batch.l_seq, np.int32)
    b.cig_off = ptr(batch.cig_off, np.uint32)
    b.cigar = ptr(batch.cigar, np.uint32)
    b.seq4 = ptr(batch.seq4, np.uint32)
    b.n_contigs = len(batch.contig_len)
    b.reads_sorted = 0
    b.contig_read_off = ptr(batch.contig_read_off, np.int64)
    b.contig_len = ptr(batch.contig_len, np.int32)
    b.contig_slot = ptr(batch.contig_slot, np.int64)
    b.n_complex = 0
    b.complex_idx = None
    b.evt_off = None
    return b


def pileup(batch, counts=None):
    """Sequential CIGAR walk over every read (kindel.py:40-81).  Raises like the reference."""
    lib = _load()
    keep = []
    b = _struct(batch, keep)
    n_slots = int(batch.n_slots)
    if counts is None:
        counts = np.zeros((NCOL, n_slots), dtype=np.int32)
    n_ins_ops = int(((np.asarray(batch.cigar) & 15) == 1).sum())
    events = np.zeros((max(n_ins_ops, 1), 4), dtype=np.int32)
    n_evt = C.c_int64(0)
    diag = _Diag()
    rc = lib.oracle_pileup(C.byref(b), counts.ctypes.data, n_slots, events.ctypes.data, C.byref(n_evt),
                           C.byref(diag))
    if rc == 10:
        raise IndexError("read %d (op %d) walks off its contig or its SEQ" % (diag.read, diag.op_index))
    if rc == 11:
        raise KeyError(NIBBLES[diag.nibble])
    return counts, events[: n_evt.value]


def _min_depth_ceil(min_depth):
    """`depth < min_depth` (reference kindel.py:415) as `depth < ceil(min_depth)` over int64.  Written out here
    rather than taken from the engine, so the oracle stays an independent side of the comparison: nan never
    calls N; +-inf and values beyond int64 clamp to +-2**62, far outside any depth sum."""
    md = float(min_depth)
    if md != md:
        return -(2 ** 62)
    return int(math.ceil(min(max(md, -2.0 ** 62), 2.0 ** 62)))


def vote(counts, min_depth=1):
    lib = _load()
    counts = np.ascontiguousarray(counts, dtype=np.int32)
    n_slots = counts.shape[1]
    calls = np.zeros(n_slots, dtype=np.uint8)
    lib.oracle_vote(counts.ctypes.data, n_slots, _min_depth_ceil(min_depth), calls.ctypes.data)
    return calls


def derive(counts):
    lib = _load()
    counts = np.ascontiguousarray(counts, dtype=np.int32)
    n_slots = counts.shape[1]
    out = np.zeros((5, n_slots), dtype=np.int32)
    lib.oracle_derive(counts.ctypes.data, n_slots, out.ctypes.data)
    return out
