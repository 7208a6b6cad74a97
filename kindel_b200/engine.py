"""Device side of the pileup/consensus engine: torch tensors as buffers, kernels through the C ABI.

PyTorch is used for device memory, streams and (in `distributed.py`) the NCCL process group only;
every count and every vote is computed by the hand-written sm_100a kernels in
`kindel_b200/csrc/` reached through `libkindel_b200.so` (include/kindel_b200.h).  There is no CPU
implementation behind these functions: without a CUDA device they raise.

    upload(batch)              ReadBatch (host numpy) -> DeviceBatch (device tensors + kdl_batch)
    pileup(dbatch)             K1: count table [19, n_slots] int32 + insertion events
    vote(counts, min_depth)    K2: call byte per slot
    derive(counts)             derived depth columns [5, n_slots]
"""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass

import numpy as np
import torch

from . import _ffi
from .bamio import NIBBLES, ReadBatch


def require_cuda(device=None) -> torch.device:
    if not torch.cuda.is_available():
        raise RuntimeError(
            "kindel_b200 needs a CUDA device (B200, sm_100a): the pileup and the vote exist only as "
            "CUDA kernels and there is no CPU fallback")
    if device is None:
        device = torch.device("cuda", torch.cuda.current_device())
    return torch.device(device)


def _stream_ptr(device) -> int:
    return int(torch.cuda.current_stream(device).cuda_stream)


@dataclass
class DeviceBatch:
    host: ReadBatch
    device: torch.device
    tensors: dict
    struct: _ffi.KdlBatch

    @property
    def n_slots(self) -> int:
        return self.host.n_slots


def make_struct(host: ReadBatch, ptr: dict) -> _ffi.KdlBatch:
    s = _ffi.KdlBatch()
    s.n_reads = host.n_reads
    s.seq4_words = int(host.seq4.shape[0])
    s.ref_start = ptr["ref_start"]
    s.seq_off = ptr["seq_off"]
    s.l_seq = ptr["l_seq"]
    s.seq4 = ptr["seq4"]
    s.n_contigs = host.n_contigs
    s.reads_sorted = 1 if host.reads_sorted else 0
    s.max_simple_len = int(host.max_simple_len)
    s.reach_right = int(host.reach_right)
    s.reach_left = int(host.reach_left)
    s.contig_read_off = ptr["contig_read_off"]
    s.contig_len = ptr["contig_len"]
    s.contig_slot = ptr["contig_slot"]
    s.n_complex = host.n_complex
    s.n_hard = host.n_hard
    s.complex_idx = ptr["complex_idx"] if host.n_complex else None
    s.hard_idx = ptr["hard_idx"] if host.n_hard else None
    s.tile_index = ptr.get("tile_index")
    return s


_FIELDS = ("ref_start", "seq_off", "l_seq", "seq4", "contig_read_off", "contig_len", "contig_slot", "complex_idx",
           "hard_idx")


def host_struct(host: ReadBatch):
    """kdl_batch over HOST pointers (for the kdl_ctx_* entry points).  Returns (struct, keepalive)."""
    keep = {f: np.ascontiguousarray(getattr(host, f)) for f in _FIELDS}
    ptr = {f: (a.ctypes.data if a.size else None) for f, a in keep.items()}
    return make_struct(host, ptr), keep


def upload(host: ReadBatch, device=None, non_blocking: bool = False) -> DeviceBatch:
    device = require_cuda(device)
    tensors = {}
    for f in _FIELDS:
        a = np.ascontiguousarray(getattr(host, f))
        if a.dtype == np.uint32:  # torch has no first-class uint32 arithmetic; the bits are what matter
            a = a.view(np.int32)
        t = torch.from_numpy(a) if a.size else torch.zeros(4, dtype=torch.from_numpy(a).dtype)
        tensors[f] = t.to(device, non_blocking=non_blocking)
    # scratch for the tile index kdl_pileup builds on the device (K0)
    tensors["tile_index"] = torch.empty(8 * (host.n_slots // _ffi.KDL_TILE), dtype=torch.int32, device=device)
    ptr = {f: int(t.data_ptr()) for f, t in tensors.items()}
    return DeviceBatch(host=host, device=device, tensors=tensors, struct=make_struct(host, ptr))


def raise_like_reference(status: int, read: int, nibble: int, op_index: int):
    if status == _ffi.KDL_ERR_KEY:
        exc = KeyError(NIBBLES[nibble])  # e.g. KeyError('R'): kindel.py:52,72,79
    else:
        exc = IndexError("list index out of range (read %d, CIGAR op %d walks off its contig or its SEQ)"
                         % (read, op_index))
    exc.kdl_read = int(read)  # which read of the batch raised (the sharded driver orders errors by it)
    raise exc


class CountTable:
    """A count table [19, n_slots] that is REUSED across pileups without being memset.

    It remembers which slot range earlier pileups may have dirtied and whether the non-weight
    columns (5..18: indels, clips -- only complex reads write them) are dirty, and asks the kernels
    to overwrite / zero exactly that (KDL_PILEUP_FRESH_WEIGHTS / KDL_PILEUP_ZERO_REST) instead of
    clearing 76 bytes per slot every time."""

    def __init__(self, n_slots: int, device, tensor: torch.Tensor = None):
        self.n_slots = n_slots
        self.device = device
        self.t = tensor if tensor is not None else torch.zeros((_ffi.KDL_NCOL, n_slots), dtype=torch.int32,
                                                                device=device)
        self.dirty = None        # (lo, hi) slot range holding counts of an earlier pileup
        self.dirty_rest = False  # columns 5..18 non-zero somewhere inside `dirty`


def _tile_align(lo: int, hi: int, n_slots: int):
    t = _ffi.KDL_TILE
    return max(0, lo // t * t), min(n_slots, (hi + t - 1) // t * t)


def pileup(dbatch: DeviceBatch, counts: torch.Tensor = None, check: bool = True, table: CountTable = None,
           slot_range=None):
    """K1.  Returns (counts int32[19, n_slots], events int32[n_events, 4]) on the device.

    counts=<tensor>  accumulate into a table the caller zeroed (several batches / shards may add up).
    table=<CountTable>  fresh result in a reused table: nothing is memset, the kernels overwrite the
                     weight columns and zero the others only if an earlier pileup dirtied them.
                     slot_range = (lo, hi) bounds what the batch can touch (default: everything).
    With check=True the error flag is read back (one 16-byte D2H) and, if set, the exact first
    offending read is located on the device and the reference's exception is raised."""
    lib = _ffi.load()
    dev = dbatch.device
    n_slots = dbatch.n_slots
    with torch.cuda.device(dev):
        # scratch that lives with the batch: the insertion-event rows and the 16-byte error flag
        events = dbatch.tensors.get("_events")
        if events is None:
            events = dbatch.tensors["_events"] = torch.empty((max(dbatch.host.n_events, 1), 4), dtype=torch.int32,
                                                             device=dev)
            dbatch.tensors["_flag"] = torch.zeros(4, dtype=torch.int32, device=dev)
        flag = dbatch.tensors["_flag"]
        if check:
            flag.zero_()  # unchecked calls (hot loops) never read it
        if table is not None:
            counts = table.t
            lo, hi = slot_range if slot_range is not None else (0, n_slots)
            if table.dirty is not None:
                lo, hi = min(lo, table.dirty[0]), max(hi, table.dirty[1])
            lo, hi = _tile_align(lo, hi, n_slots)
            flags = _ffi.KDL_PILEUP_FRESH_WEIGHTS | (_ffi.KDL_PILEUP_ZERO_REST if table.dirty_rest else 0)
            rc = lib.kdl_pileup_range(C.byref(dbatch.struct), counts.data_ptr(), n_slots, lo, hi, flags,
                                      events.data_ptr(), flag.data_ptr(), _stream_ptr(dev))
            table.dirty = (lo, hi)
            table.dirty_rest = dbatch.host.n_complex > 0
        else:
            if counts is None:
                counts = torch.zeros((_ffi.KDL_NCOL, n_slots), dtype=torch.int32, device=dev)
            rc = lib.kdl_pileup(C.byref(dbatch.struct), counts.data_ptr(), n_slots, events.data_ptr(),
                                flag.data_ptr(), _stream_ptr(dev))
        _ffi.check(rc, "kdl_pileup")
        if check and int(flag[0].item()) != 0:
            diagnose_and_raise(dbatch)
    return counts, events[: dbatch.host.n_events]


def diagnose_and_raise(dbatch: DeviceBatch):
    lib = _ffi.load()
    dev = dbatch.device
    diag = torch.zeros(6, dtype=torch.int32, device=dev)  # sizeof(kdl_diag) == 24
    rc = lib.kdl_diagnose(C.byref(dbatch.struct), diag.data_ptr(), _stream_ptr(dev))
    _ffi.check(rc, "kdl_diagnose")
    raw = diag.cpu().numpy().tobytes()
    d = _ffi.KdlDiag.from_buffer_copy(raw)
    if d.status:
        raise_like_reference(d.status, d.read, d.nibble, d.op_index)
    raise RuntimeError("pileup raised its error flag but no offending read was found")


MIN_DEPTH_CLAMP = 2 ** 62


def min_depth_ceil(min_depth) -> int:
    """The int64 the vote kernels compare an integer depth with: `depth < min_depth` (kindel.py:415) is
    `depth < ceil(min_depth)`.  nan compares false with everything, so it never calls N; +-inf and finite values
    beyond int64 are clamped to +-2**62.  Depth sums are at most 5 * (2**31 - 1), so the clamp changes no answer."""
    md = float(min_depth)
    if math.isnan(md):
        return -MIN_DEPTH_CLAMP
    if md >= MIN_DEPTH_CLAMP:
        return MIN_DEPTH_CLAMP
    if md <= -MIN_DEPTH_CLAMP:
        return -MIN_DEPTH_CLAMP
    return int(math.ceil(md))


def vote(counts: torch.Tensor, min_depth=1, out: torch.Tensor = None) -> torch.Tensor:
    """K2.  counts int32[>=7, n_slots] (contiguous) -> calls uint8[n_slots] (`out` reuses a buffer)."""
    lib = _ffi.load()
    dev = counts.device
    n_slots = counts.shape[1]
    with torch.cuda.device(dev):
        calls = out if out is not None else torch.empty(n_slots, dtype=torch.uint8, device=dev)
        rc = lib.kdl_vote(counts.data_ptr(), n_slots, min_depth_ceil(min_depth), calls.data_ptr(),
                          _stream_ptr(dev))
        _ffi.check(rc, "kdl_vote")
    return calls


def derive(counts: torch.Tensor) -> torch.Tensor:
    """Derived columns [5, n_slots]: consensus_depth, clip_start_depth, clip_end_depth, clip_depth,
    acgt_depth (kindel.py:83-96, :450)."""
    lib = _ffi.load()
    dev = counts.device
    n_slots = counts.shape[1]
    with torch.cuda.device(dev):
        out = torch.empty((5, n_slots), dtype=torch.int32, device=dev)
        rc = lib.kdl_derive(counts.data_ptr(), n_slots, out.data_ptr(), _stream_ptr(dev))
        _ffi.check(rc, "kdl_derive")
    return out


def cdr_flags(counts: torch.Tensor, slot_lo: int, slot_hi: int, clip_decay_threshold: float):
    """K4: (flags uint8[slot_hi - slot_lo], bases uint8[...]) on the host for slots [slot_lo, slot_hi): the
    --realign predicates (kindel.py:182-185,202,243-246,256), 2 bytes per slot instead of the 76-byte table row."""
    lib = _ffi.load()
    dev = counts.device
    n_slots = counts.shape[1]
    with torch.cuda.device(dev):
        flags = torch.empty(n_slots, dtype=torch.uint8, device=dev)
        bases = torch.empty(n_slots, dtype=torch.uint8, device=dev)
        rc = lib.kdl_cdr_flags(counts.data_ptr(), n_slots, int(slot_lo), int(slot_hi), float(clip_decay_threshold),
                               flags.data_ptr(), bases.data_ptr(), _stream_ptr(dev))
        _ffi.check(rc, "kdl_cdr_flags")
    return flags[slot_lo:slot_hi].cpu().numpy(), bases[slot_lo:slot_hi].cpu().numpy()


def assemble(calls: torch.Tensor, host: ReadBatch, ins_slots: np.ndarray, ins_strings):
    """K5: consensus text of every contig from the device call bytes.  ins_slots (ascending) / ins_strings: the
    chosen insertion string of every slot whose call carries change 'I'.  Returns a list of str, one per contig."""
    lib = _ffi.load()
    dev = calls.device
    n_slots = int(calls.shape[0])
    enc = [x.encode("ascii") for x in ins_strings]
    ins_off = np.zeros(len(enc) + 1, dtype=np.uint32)
    if enc:
        ins_off[1:] = np.cumsum([len(x) for x in enc])
    blob = np.frombuffer(b"".join(enc) or b"\0", dtype=np.uint8)
    with torch.cuda.device(dev):
        def put(a):
            a = np.ascontiguousarray(a)
            return torch.from_numpy(a.view(np.int32) if a.dtype == np.uint32 else a).to(dev)

        t_slot = put(np.asarray(host.contig_slot, dtype=np.int64))
        t_len = put(np.asarray(host.contig_len, dtype=np.int32))
        t_is = put(np.asarray(ins_slots, dtype=np.int64) if len(enc) else np.zeros(1, dtype=np.int64))
        t_io = put(ins_off)
        t_ib = put(blob.copy())
        sums = torch.empty(int(lib.kdl_assemble_scratch_words(n_slots)), dtype=torch.int32, device=dev)
        offsets = torch.empty(n_slots + 1, dtype=torch.int32, device=dev)
        out = torch.empty(n_slots + int(ins_off[-1]) + 16, dtype=torch.uint8, device=dev)
        rc = lib.kdl_assemble(calls.data_ptr(), n_slots, t_slot.data_ptr(), t_len.data_ptr(), host.n_contigs,
                              t_is.data_ptr(), t_io.data_ptr(), t_ib.data_ptr(), len(enc), sums.data_ptr(),
                              offsets.data_ptr(), out.data_ptr(), _stream_ptr(dev))
        _ffi.check(rc, "kdl_assemble")
        starts = torch.from_numpy(np.asarray(host.contig_slot, dtype=np.int64)).to(dev)
        ends = starts + torch.from_numpy(np.asarray(host.contig_len, dtype=np.int64)).to(dev)
        lo = offsets[starts].cpu().numpy().astype(np.int64) & 0xFFFFFFFF
        hi = offsets[ends].cpu().numpy().astype(np.int64) & 0xFFFFFFFF
        total = int(offsets[n_slots].item()) & 0xFFFFFFFF
        text = out[:total].cpu().numpy().tobytes()
    return [text[a:b].decode("ascii") for a, b in zip(lo.tolist(), hi.tolist())]


class HostContext:
    """kdl_ctx_*: host buffers in, host buffers out (the path a non-CUDA host program binds)."""

    def __init__(self, device: int = 0):
        self._lib = _ffi.load()
        h = C.c_void_p()
        rc = self._lib.kdl_ctx_create(int(device), C.byref(h))
        _ffi.check(rc, "kdl_ctx_create")
        self._h = h

    def close(self):
        if self._h:
            self._lib.kdl_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def consensus(self, host: ReadBatch, min_depth=1, calls_out=None, counts_out=None, events_out=None,
                  struct=None):
        """Runs H2D + K1 + K2 + D2H.  Returns calls (numpy uint8[n_slots])."""
        if struct is None:
            struct, keep = host_struct(host)
        if calls_out is None:
            calls_out = np.empty(host.n_slots, dtype=np.uint8)
        diag = _ffi.KdlDiag()
        rc = self._lib.kdl_ctx_consensus(
            self._h, C.byref(struct), host.n_slots, host.n_events, min_depth_ceil(min_depth),
            calls_out.ctypes.data, counts_out.ctypes.data if counts_out is not None else None,
            events_out.ctypes.data if (events_out is not None and host.n_events) else None, C.byref(diag))
        if rc in (_ffi.KDL_ERR_INDEX, _ffi.KDL_ERR_KEY):
            raise_like_reference(rc, diag.read, diag.nibble, diag.op_index)
        _ffi.check(rc, "kdl_ctx_consensus")
        return calls_out

    def last_timing(self):
        a, b, c = C.c_float(), C.c_float(), C.c_float()
        self._lib.kdl_ctx_last_timing(self._h, C.byref(a), C.byref(b), C.byref(c))
        return {"h2d_ms": a.value, "kernel_ms": b.value, "d2h_ms": c.value}
