"""The kernels that turn a finished count table into the answer -- K2 / K2p / K2x (vote), K2d (derived columns),
K4 (--realign flags) and K5 (consensus text) -- on adversarial tables (tests/table_cases.py), against

  * the unmodified reference's own results on those tables (tests/golden/table_runs.json.gz,
    oracle/make_table_golden.py), and
  * a plain numpy / float64 restatement of the reference's per-position expressions (below), which a CPU test first
    checks against the stored results and which then serves for tables too large to store.

Every kernel test runs on two backends: the emulator (tests/emu/, the kernels' source compiled for the host; always)
and the library on the GPU (`-m gpu`)."""
from __future__ import annotations

import ctypes as C
import gzip
import json
import math
import os
import random
from types import SimpleNamespace

import numpy as np
import pytest

import emu_harness as E
import table_cases as T
from kindel_b200 import kindel as K

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "table_runs.json.gz")
_LETTERS = "ACGTN"
_ORDER = np.array([0, 3, 2, 1, 4])  # the reference's dict order A,T,G,C,N as table columns A,C,G,T,N


@pytest.fixture(scope="module")
def golden():
    with gzip.open(GOLDEN, "rt") as fh:
        return json.load(fh)


@pytest.fixture(scope="module")
def cases():
    return [T.table_case(s) for s in range(T.N_CASES)]


# ------------------------------------------------------------------------------------------------ restatement
def first_max(w5):
    """consensus(w) (kindel.py:369-381) of every column of a [5, n] A,C,G,T,N block: (column of the first maximum in
    A,T,G,C,N order, or N when all are zero; its count; tie = another key holds the same non-zero count)."""
    stacked = np.asarray(w5, dtype=np.int64)[_ORDER]
    freq = stacked.max(axis=0)
    code = _ORDER[np.argmax(stacked, axis=0)]
    empty = stacked.sum(axis=0) == 0
    code = np.where(empty, 4, code)
    freq = np.where(empty, 0, freq)
    tie = (freq != 0) & ((stacked == freq).sum(axis=0) > 1)
    return code, freq, tie


def restate_calls(counts, min_depth):
    """consensus_sequence's per-position decisions (kindel.py:402-424) for every slot of the table, as call bytes:
    bits 0-2 the emitted base (N for a tie), bits 4-5 the change (0 none, 1 D, 2 N, 3 I).  The slot after the last
    one counts as depth 0, as the reference's IndexError branch does at a contig's end."""
    c = np.asarray(counts, dtype=np.float64)
    depth = c[0] + c[1] + c[2] + c[3]  # N is not part of aligned_depth (kindel.py:404)
    depth_next = np.append(depth[1:], 0.0)
    threshold = depth * 0.5
    indel_threshold = np.minimum(threshold, depth_next * 0.5)
    is_d = c[5] > threshold
    is_n = ~is_d & (depth < min_depth)
    is_i = ~is_d & ~is_n & (c[6] > indel_threshold)
    code, _, tie = first_max(counts[0:5])
    base = np.where(tie | is_d | is_n, 4, code)
    change = np.select([is_d, is_n, is_i], [1, 2, 3], 0)
    return (change << 4 | base).astype(np.uint8)


def restate_derive(counts):
    """consensus_depth, clip_start_depth, clip_end_depth, clip_depth, ACGT depth (kindel.py:83-96, :450)."""
    c = np.asarray(counts, dtype=np.int64)
    _, freq, _ = first_max(c[0:5])
    csd, ced = c[9:13].sum(axis=0), c[14:18].sum(axis=0)
    return np.stack([freq, csd, ced, csd + ced, c[0:4].sum(axis=0)]).astype(np.int32)


def restate_cdr(counts, lo, hi, decay):
    """The --realign predicates (kindel.py:182-185, 202, 243-246, 256) in K4's byte layout."""
    c = np.asarray(counts[:, lo:hi], dtype=np.int64)
    tot = c[0:5].sum(axis=0) + c[5]  # sum(w.values()) + deletions: all five keys
    flags = np.zeros(hi - lo, dtype=np.uint8)
    bases = np.zeros(hi - lo, dtype=np.uint8)
    for d, c0 in enumerate((9, 14)):
        cd = c[c0:c0 + 4].sum(axis=0)  # clip depth: A,C,G,T (kindel.py:90-95)
        dominant = cd / (tot + 1) > 0.5
        extend = cd > tot * decay
        flags |= (dominant.astype(np.uint8) << (2 * d)) | (extend.astype(np.uint8) << (2 * d + 1))
        bases |= first_max(c[c0:c0 + 5])[0].astype(np.uint8) << (4 * d)
    return flags, bases


def restate_text(calls, contig_slot, contig_len, ins_text):
    """K5's text: per contig, per position, nothing for D, else the insertion string (I) and the base letter."""
    out = []
    for s0, L in zip(np.asarray(contig_slot).tolist(), np.asarray(contig_len).tolist()):
        parts = []
        for s in range(s0, s0 + L):
            c = int(calls[s])
            change = (c >> 4) & 3
            if change == 1:
                continue
            if change == 3:
                parts.append(ins_text[s])
            parts.append(_LETTERS[min(c & 7, 4)])
        out.append("".join(parts))
    return out


def dict_choice(items):
    """The string consensus_sequence prints for an 'I' call (kindel.py:420-421): the first most frequent inserted
    string in first-seen order, lower-cased, or N for a tie."""
    best, freq = None, 0
    for s, n in items:
        if n > freq:
            best, freq = s, n
    tie = sum(1 for s, n in items if n == freq) > 1
    return "N" if tie else best.lower()


def changes_text(calls):
    return "".join("-DNI"[(int(c) >> 4) & 3] for c in calls)


def regions_from_flags(flags, bases, mask_ends):
    """Regions as cdrps_from_device builds them from K4's bytes."""
    n = flags.shape[0]
    keep = ~K._masked(n, mask_ends)
    chars = np.frombuffer(b"ACGTN", dtype=np.uint8)
    fwd = K._start_regions(n, ((flags & 1) != 0) & keep, (flags & 2) != 0, chars[np.minimum(bases & 7, 4)])
    rev = K._end_regions(n, ((flags & 4) != 0) & keep, (flags & 8) != 0, chars[np.minimum((bases >> 4) & 7, 4)])
    return [list(r) for r in fwd], [list(r) for r in rev]


# ------------------------------------------------------------------------------------------------ backends
def exchange_grid(slice_lo, slice_hi):
    """CTAs kdl_exchange_vote launches for a slice (below its cap of 8 CTAs per SM, which these slices never reach)."""
    return max(1, ((slice_hi - slice_lo) // 4 + 255) // 256)


def chunk_ends(slice_lo, slice_hi, grid):
    """End slot of every CTA's chunk of a slice in vote_exchange_kernel (whole warps of quads per CTA)."""
    quads = (slice_hi - slice_lo + 3) >> 2
    per_cta = ((quads + grid - 1) // grid + 31) & ~31
    last = (quads + 31) & ~31
    return [slice_lo + 4 * min(b * per_cta + per_cta, last) for b in range(grid) if b * per_cta < last]


class Emu:
    name = "emu"

    def vote(self, counts, md):
        return E.vote(counts, md)

    def derive(self, counts):
        return E.derive(counts)

    def cdr_flags(self, counts, lo, hi, decay):
        return E.cdr_flags(counts, lo, hi, decay)

    def assemble(self, calls, contig_slot, contig_len, ins_slots, ins_strings):
        return E.assemble(calls, contig_slot, contig_len, ins_slots, ins_strings)

    def vote_peers(self, tables, feet, lo, hi, md):
        return E.vote_peers(tables, feet, lo, hi, md, want_reduced=True)

    def exchange(self, tables, feet, slices, md):
        world, n_slots = len(tables), tables[0].shape[1]
        flags = {k: [np.zeros(16, dtype=np.int32) for _ in range(world)] for k in ("ready", "done")}
        flags["counter"] = [np.zeros(1, dtype=np.int32) for _ in range(world)]
        calls = [np.full(n_slots, 0xEE, dtype=np.uint8) for _ in range(world)]
        # the emulator launches one grid for every rank: rank 0's, so its slice is cut into the chunks
        # kdl_exchange_vote would cut it into (any grid is a valid cut of the other slices)
        grid = exchange_grid(*slices[0])
        E.exchange_epoch([np.ascontiguousarray(t) for t in tables], feet, slices, calls, flags, 1, md, grid=grid)
        return calls


class Gpu:
    name = "gpu"

    def __init__(self):
        import torch

        from kindel_b200 import _ffi, engine

        self.torch, self.engine, self.ffi = torch, engine, _ffi
        self.dev = torch.device("cuda", torch.cuda.current_device())

    def _t(self, a):
        return self.torch.from_numpy(np.ascontiguousarray(a)).to(self.dev)

    def vote(self, counts, md):
        return self.engine.vote(self._t(counts), md).cpu().numpy()

    def derive(self, counts):
        return self.engine.derive(self._t(counts)).cpu().numpy()

    def cdr_flags(self, counts, lo, hi, decay):
        return self.engine.cdr_flags(self._t(counts), lo, hi, decay)

    def assemble(self, calls, contig_slot, contig_len, ins_slots, ins_strings):
        host = SimpleNamespace(contig_slot=np.asarray(contig_slot, dtype=np.int64),
                               contig_len=np.asarray(contig_len, dtype=np.int32), n_contigs=len(contig_slot))
        return self.engine.assemble(self._t(calls), host, np.asarray(ins_slots, dtype=np.int64), ins_strings)

    def vote_peers(self, tables, feet, lo, hi, md):
        n, n_slots = len(tables), tables[0].shape[1]
        dt = [self._t(t) for t in tables]
        calls = self.torch.full((n_slots,), 0xEE, dtype=self.torch.uint8, device=self.dev)
        reduced = self.torch.zeros((7, n_slots), dtype=self.torch.int32, device=self.dev)
        ptrs = (C.c_void_p * n)(*[t.data_ptr() for t in dt])
        flo = (C.c_int64 * n)(*[f[0] for f in feet])
        fhi = (C.c_int64 * n)(*[f[1] for f in feet])
        rc = self.ffi.load().kdl_vote_peers_sparse(ptrs, flo, fhi, n, n_slots, lo, hi, self.engine.min_depth_ceil(md),
                                                   calls.data_ptr(), reduced.data_ptr(),
                                                   int(self.torch.cuda.current_stream(self.dev).cuda_stream))
        self.ffi.check(rc, "kdl_vote_peers_sparse")
        return calls.cpu().numpy(), reduced.cpu().numpy()

    def exchange(self, tables, feet, slices, md):
        """K2x + K2g for every rank inside this process: the ranks' blocks are allocations of one device, and the
        kernels are issued in an order that never has to wait on a flag."""
        torch, ffi = self.torch, self.ffi
        lib = ffi.load()
        st = int(torch.cuda.current_stream(self.dev).cuda_stream)
        world, S = len(tables), tables[0].shape[1]
        table_bytes = 19 * S * 4
        calls_off, flags_off = table_bytes, table_bytes + S
        blocks = [torch.zeros(flags_off + 256, dtype=torch.uint8, device=self.dev) for _ in range(world)]
        for blk, t in zip(blocks, tables):
            blk[:table_bytes].view(torch.int32).view(19, S).copy_(self._t(t))
        xs = []
        for r in range(world):
            x = ffi.KdlExchange()
            x.n_ranks, x.rank = world, r
            for p, blk in enumerate(blocks):
                base = blk.data_ptr()
                x.tables[p], x.calls[p] = base, base + calls_off
                x.ready[p], x.done[p] = base + flags_off, base + flags_off + 64
                x.foot_lo[p], x.foot_hi[p] = feet[p]
                x.slice_lo[p], x.slice_hi[p] = slices[p]
            x.counter = blocks[r].data_ptr() + flags_off + 128
            xs.append(x)
        md_ceil = self.engine.min_depth_ceil(md)
        for r in range(world):
            ffi.check(lib.kdl_exchange_signal(C.byref(xs[r]), 1, st), "kdl_exchange_signal")
        for r in range(world):
            ffi.check(lib.kdl_exchange_vote(C.byref(xs[r]), S, md_ceil, 1, st), "kdl_exchange_vote")
        for r in range(world):
            ffi.check(lib.kdl_exchange_wait(C.byref(xs[r]), 1, st), "kdl_exchange_wait")
        torch.cuda.synchronize()
        return [blk[calls_off:calls_off + S].cpu().numpy() for blk in blocks]


@pytest.fixture(scope="module", params=["emu", pytest.param("gpu", marks=pytest.mark.gpu)])
def be(request):
    if request.param == "emu":
        if not E.available():
            pytest.skip("needs g++ and the CUDA headers")
        return Emu()
    return Gpu()


# ------------------------------------------------------------------------------------------------ helpers
def insertion_inputs(calls, ins):
    """(ascending slots, strings) of every 'I' call that has an insertion dict -- the extra slot behind a contig
    included, which K5 must not print."""
    slots = [s for s in np.flatnonzero(((calls >> 4) & 3) == 3).tolist() if s in ins]
    return slots, [dict_choice(list(ins[s].items())) for s in slots]


def packed(cases, layout):
    rng = random.Random(5)
    return T.pack(cases, rng, align=1024 if layout == "aligned" else None)


def split_tables(counts, feet, rng):
    """Peer tables whose sum is `counts`, table p zero outside feet[p]; each slot's counts shared at random between
    the tables that cover it."""
    n_slots = counts.shape[1]
    tables = [np.zeros_like(counts) for _ in feet]
    rest = counts.astype(np.int64)
    slots = np.arange(n_slots)
    for p, (lo, hi) in enumerate(feet):
        cover = (slots >= lo) & (slots < hi)
        later = np.zeros(n_slots, dtype=bool)
        for lo2, hi2 in feet[p + 1:]:
            later |= (slots >= lo2) & (slots < hi2)
        take = np.where(later, (rest * rng.random(rest.shape)).astype(np.int64), rest)
        take[:, ~cover] = 0
        tables[p] = take.astype(np.int32)
        rest = rest - take
    assert not rest.any(), "the footprints must cover every non-zero slot"
    return tables


# ------------------------------------------------------------------------------------------------ CPU: restatement
def test_restatement_equals_the_reference(golden, cases):
    """The numpy restatement against what the reference returned on the same tables: sequences and changes for
    every min_depth, CDR regions for every (decay, mask_ends), consensus() of every position."""
    assert sorted(golden["cases"], key=int) == [str(s) for s in range(T.N_CASES)]
    for seed, case in enumerate(cases):
        want = golden["cases"][str(seed)]
        L, counts = case["L"], case["counts"]
        assert want["L"] == L
        code, freq, tie = first_max(counts[0:5, :L])
        assert "".join(_LETTERS[k] for k in code) == want["base"], seed
        assert freq.tolist() == want["freq"], seed
        assert "".join("1" if t else "0" for t in tie) == want["tie"], seed
        ins = {k: dict(v) for k, v in case["insertions"].items()}
        for name, md in T.MIN_DEPTHS:
            calls = restate_calls(counts, md)
            slots, strings = insertion_inputs(calls, ins)
            seq = restate_text(calls, [0], [L], dict(zip(slots, strings)))[0]
            assert [seq, changes_text(calls[:L])] == want["consensus"][name], (seed, name)
        for decay, mask in T.CDR_OPTIONS:
            flags, bases = restate_cdr(counts, 0, L, decay)
            fwd, rev = regions_from_flags(flags, bases, mask)
            w = want["cdr"][T.cdr_key(decay, mask)]
            assert fwd == w["start"] and rev == w["end"], (seed, decay, mask)


def test_cases_sit_on_the_boundaries(cases):
    """The generator does plant what the kernels can get wrong (a guard against a quietly weakened generator)."""
    seen = {"ins_eq": 0, "ins_eq1": 0, "del_eq": 0, "del_eq1": 0, "tie": 0, "nonly": 0, "dom_eq": 0, "ext_eq": 0,
            "lane31": 0, "cta": 0}
    for case in cases:
        c = case["counts"].astype(np.int64)
        d = c[0:4].sum(axis=0)
        dn = np.append(d[1:], 0)
        thr = np.minimum(d, dn)
        lookahead = (dn < d) & (d > 0)
        seen["ins_eq"] += int(((2 * c[6] == thr) & lookahead & (thr > 0)).sum())
        seen["ins_eq1"] += int(((2 * c[6] == thr + 1) & lookahead).sum())
        seen["del_eq"] += int(((2 * c[5] == d) & (d > 0)).sum())
        seen["del_eq1"] += int((2 * c[5] == d + 1).sum())
        seen["tie"] += int(first_max(c[0:5])[2].sum())
        seen["nonly"] += int(((d == 0) & (c[4] > 0)).sum())
        tot = c[0:5].sum(axis=0) + c[5]
        for c0 in (9, 14):
            cd = c[c0:c0 + 4].sum(axis=0)
            seen["dom_eq"] += int((2 * cd == tot + 1).sum())
            seen["ext_eq"] += int(sum(((cd == tot * x) & (tot > 0)).sum() for x in T.DECAYS))
        L = case["L"]
        idx = np.arange(L)
        seen["lane31"] += int((((idx % 128) == 127) & (2 * c[6, :L] >= thr[:L]) & lookahead[:L]).sum())
        seen["cta"] += int((((idx % 1024) == 1023) & lookahead[:L]).sum())
    assert all(v > 0 for v in seen.values()), seen
    assert seen["ins_eq"] > 50 and seen["ins_eq1"] > 50 and seen["dom_eq"] > 20 and seen["ext_eq"] > 20, seen


def test_min_depth_ceil_maps_every_float():
    from kindel_b200 import engine
    from oracle import coracle

    big = 2 ** 62
    for conv in (engine.min_depth_ceil, coracle._min_depth_ceil):
        assert conv(math.nan) == -big  # `depth < nan` is False: never N
        assert conv(math.inf) == big and conv(1e19) == big and conv(2.0 ** 63) == big
        assert conv(-math.inf) == -big and conv(-1e19) == -big
        assert conv(2.5) == 3 and conv(2) == 2 and conv(0) == 0 and conv(-0.5) == 0 and conv(7) == 7


@pytest.mark.parametrize("name", [name for name, _ in T.MIN_DEPTHS])
def test_oracle_vote_min_depth_edges(cases, name):
    """The C oracle's vote (the other side of the pileup comparisons) on every min_depth."""
    from oracle import coracle

    md = dict(T.MIN_DEPTHS)[name]

    counts, _, _, _ = packed(cases, "tight")
    np.testing.assert_array_equal(coracle.vote(counts, md), restate_calls(counts, md))


# ------------------------------------------------------------------------------------------------ K2 + K2d + K5
@pytest.mark.parametrize("layout", ["aligned", "tight"])
def test_vote_derive_and_text_equal_the_reference(be, golden, cases, layout):
    """K2 on the packed golden tables (contigs at multiples of 1024, or at arbitrary slots), for every min_depth:
    call bytes == restatement on every slot; per contig, K5's text and the changes == the reference's.  K2d ==
    restatement and the reference's consensus() counts."""
    counts, cslot, clen, ins = packed(cases, layout)
    derived = be.derive(counts)
    np.testing.assert_array_equal(derived, restate_derive(counts))
    for seed, (s0, L) in enumerate(zip(cslot.tolist(), clen.tolist())):
        assert derived[0, s0:s0 + L].tolist() == golden["cases"][str(seed)]["freq"]
    for name, md in T.MIN_DEPTHS:
        calls = be.vote(counts, md)
        np.testing.assert_array_equal(calls, restate_calls(counts, md), err_msg="min_depth %s" % name)
        slots, strings = insertion_inputs(calls, ins)
        texts = be.assemble(calls, cslot, clen, slots, strings)
        for seed, (s0, L) in enumerate(zip(cslot.tolist(), clen.tolist())):
            want = golden["cases"][str(seed)]["consensus"][name]
            assert [texts[seed], changes_text(calls[s0:s0 + L])] == want, (seed, name)


# ------------------------------------------------------------------------------------------------ K4
def test_cdr_flags_equal_the_reference(be, golden, cases):
    """K4 == restatement bit for bit on the whole table for every decay; per contig (its slot range, as
    cdrps_from_device asks for it), the regions built from K4's bytes == the reference's Regions."""
    counts, cslot, clen, _ = packed(cases, "tight")
    n = counts.shape[1]
    for decay in T.DECAYS:
        flags, bases = be.cdr_flags(counts, 0, n, decay)
        want_f, want_b = restate_cdr(counts, 0, n, decay)
        np.testing.assert_array_equal(flags, want_f, err_msg="decay %r" % decay)
        np.testing.assert_array_equal(bases, want_b, err_msg="decay %r" % decay)
    for decay, mask in T.CDR_OPTIONS:
        for seed, (s0, L) in enumerate(zip(cslot.tolist(), clen.tolist())):
            flags, bases = be.cdr_flags(counts, s0, s0 + L, decay)
            fwd, rev = regions_from_flags(flags, bases, mask)
            w = golden["cases"][str(seed)]["cdr"][T.cdr_key(decay, mask)]
            assert fwd == w["start"] and rev == w["end"], (seed, decay, mask)


# ------------------------------------------------------------------------------------------------ K2p + K2x
def _slice_cuts(n_slots, k, rng):
    """k slices of [0, n_slots): bounds multiples of 4, never multiples of 1024."""
    cuts = set()
    while len(cuts) < k - 1:
        c = rng.randrange(1, n_slots // 4) * 4
        if c % 1024:
            cuts.add(c)
    b = [0] + sorted(cuts) + [n_slots]
    return list(zip(b[:-1], b[1:]))


def _feet(slices, n_slots, rng):
    """Overlapping footprints (multiples of 4) around the slices, covering everything."""
    feet = []
    for lo, hi in slices:
        feet.append((max(0, lo - 4 * rng.randint(1, 40)), min(n_slots, hi + 4 * rng.randint(1, 40))))
    return feet


@pytest.mark.parametrize("n_peers", [2, 3, 4])
def test_peer_vote_equals_the_single_table(be, cases, n_peers):
    """K2p over 2-4 peer tables with overlapping footprints, on slices that are not on 1024 boundaries, with an
    insertion decided by the look-ahead at every slice's last slot: calls and `reduced` == one table's vote."""
    rng = random.Random(100 + n_peers)
    counts, _, _, _ = packed(cases, "tight")
    counts = counts.copy()
    n_slots = counts.shape[1]
    slices = _slice_cuts(n_slots, n_peers, rng)
    for lo, hi in slices[:-1]:
        T.plant_ins_boundary(rng, counts, hi - 1, rng.random() < 0.5, dn=rng.randint(1, 4))
    feet = _feet(slices, n_slots, rng)
    tables = split_tables(counts, feet, np.random.default_rng(n_peers))
    for md in (2, 0, math.nan):
        want = restate_calls(counts, md)
        np.testing.assert_array_equal(be.vote(counts, md), want)
        for lo, hi in slices:
            calls, reduced = be.vote_peers(tables, feet, lo, hi, md)
            np.testing.assert_array_equal(calls[lo:hi], want[lo:hi], err_msg="slice %d..%d" % (lo, hi))
            np.testing.assert_array_equal(reduced[:, lo:hi], counts[:7, lo:hi])


@pytest.mark.parametrize("world", [2, 3])
def test_exchange_vote_at_chunk_edges(be, cases, world):
    """K2x + K2g for every rank.  The last rank's footprint starts exactly at the end of a CTA chunk of rank 0's
    slice (chunks computed from the grid kdl_exchange_vote launches), under an insertion whose call that rank's depth
    flips: there the look-ahead of the chunk's last quad is the only read of that table.  Every rank's calls ==
    one table's vote."""
    rng = random.Random(200 + world)
    base, _, _, _ = packed(cases, "tight")
    n_slots = base.shape[1]
    slices = _slice_cuts(n_slots, world, rng)
    while slices[0][1] - slices[0][0] < 3 * 1024:
        slices = _slice_cuts(n_slots, world, rng)
    ends = [e for e in chunk_ends(*slices[0], exchange_grid(*slices[0])) if e < slices[0][1]]
    assert ends, "rank 0's slice must span several chunks"
    for e in ends[:2]:
        counts = base.copy()
        T.plant_ins_boundary(rng, counts, e - 1, True, dn=2 * rng.randint(1, 3))  # 2 ins == dn: no call
        feet = _feet(slices, n_slots, rng)
        feet[0] = (0, max(feet[0][1], e + 8))
        feet[-1] = (e, n_slots)
        tables = split_tables(counts, feet, np.random.default_rng(e))
        for p in range(world - 1):  # the depth at slot e lives in the last table only
            tables[-1][0:4, e] += tables[p][0:4, e]
            tables[p][0:4, e] = 0
        for md in (1, math.inf):
            want = restate_calls(counts, md)
            got = be.exchange(tables, feet, slices, md)
            for r in range(world):
                np.testing.assert_array_equal(got[r], want, err_msg="rank %d, chunk end %d" % (r, e))


# ------------------------------------------------------------------------------------------------ K5 shapes
def _random_calls(rng, n_slots):
    change = rng.choice(4, size=n_slots, p=[0.55, 0.2, 0.1, 0.15])
    base = rng.integers(0, 5, size=n_slots)
    return (change << 4 | base).astype(np.uint8)


def _layout(rng, n_slots, n_contigs):
    """n_contigs contigs at arbitrary slots (some of length 1), each owning L + 1 slots inside the table."""
    if n_contigs == 1:
        return np.array([3], dtype=np.int64), np.array([n_slots - 5], dtype=np.int32)
    bounds = np.sort(rng.choice(np.arange(1, n_slots - 1), size=2 * n_contigs - 1, replace=False))
    edges = np.concatenate([[0], bounds, [n_slots]])
    starts, lens = [], []
    for k in range(n_contigs):
        lo, hi = int(edges[2 * k]), int(edges[2 * k + 1])
        L = 1 if k % 7 == 3 else max(1, hi - lo - 1)
        starts.append(lo)
        lens.append(L)
    return np.array(starts, dtype=np.int64), np.array(lens, dtype=np.int32)


@pytest.mark.parametrize("n_slots,n_contigs", [(262_144, 1), (262_143, 2), (600_001, 64), (3 * 1024 + 1, 300),
                                               (5 * 1024 - 1, 300), (8 * 1024, 2)])
def test_text_shapes(be, n_slots, n_contigs):
    """K5 on random call bytes: a lone block in the scan's second round (262 144 slots), sizes around multiples of
    1024, 1-300 contigs at arbitrary slots, long insertion strings at the last slot of a CTA, 'I' calls on the extra
    slot behind every contig (never printed) and in the gaps."""
    rng = np.random.default_rng(n_slots + n_contigs)
    calls = _random_calls(rng, n_slots)
    cslot, clen = _layout(rng, n_slots, n_contigs)
    ends = cslot + clen
    calls[ends[ends < n_slots]] = 0x30 | 2
    calls[np.arange(1023, n_slots, 1024)] = 0x31
    slots = np.flatnonzero(((calls >> 4) & 3) == 3)
    strings = []
    for s in slots.tolist():
        ln = int(rng.integers(300, 3000)) if s % 1024 == 1023 else int(rng.integers(1, 6))
        strings.append("".join("acgtn"[k] for k in rng.integers(0, 5, size=ln)))
    got = be.assemble(calls, cslot, clen, slots, strings)
    want = restate_text(calls, cslot, clen, dict(zip(slots.tolist(), strings)))
    assert len(got) == len(want) == n_contigs
    for c, (g, w) in enumerate(zip(got, want)):
        assert g == w, "contig %d at slot %d, length %d" % (c, cslot[c], clen[c])


def test_text_all_deletions(be):
    calls = np.full(4096, 0x14, dtype=np.uint8)
    assert be.assemble(calls, [0, 2000], [1999, 2095], [], []) == ["", ""]


# ------------------------------------------------------------------------------------------------ large (GPU)
@pytest.mark.gpu
def test_large_tier_on_the_gpu():
    """10**7 slots with counts up to 2**24 through K2, K2d, K4 and K5 on the device, against the restatement."""
    be = Gpu()
    n_slots = 10_000_000
    counts = T.large_table(11, n_slots)
    md = 2.5
    calls = be.vote(counts, md)
    np.testing.assert_array_equal(calls, restate_calls(counts, md))
    np.testing.assert_array_equal(be.derive(counts), restate_derive(counts))
    for decay in (0.1, 1 / 3, 0.7):
        lo, hi = 12_344, n_slots - 7
        flags, bases = be.cdr_flags(counts, lo, hi, decay)
        want_f, want_b = restate_cdr(counts, lo, hi, decay)
        np.testing.assert_array_equal(flags, want_f)
        np.testing.assert_array_equal(bases, want_b)
    rng = np.random.default_rng(12)
    cslot, clen = _layout(rng, n_slots, 37)
    slots = np.flatnonzero(((calls >> 4) & 3) == 3)
    ins_char = np.frombuffer(b"acgt", dtype=np.uint8)[slots % 4]
    got = be.assemble(calls, cslot, clen, slots, [chr(x) for x in ins_char.tolist()])
    # the restatement, vectorised: each position emits [insertion char if I] [base letter], nothing for D
    change = (calls >> 4) & 3
    letters = np.frombuffer(b"ACGTN", dtype=np.uint8)[np.minimum(calls & 7, 4)]
    pair = np.zeros((n_slots, 2), dtype=np.uint8)
    pair[:, 1] = letters
    pair[slots, 0] = ins_char
    emit = np.stack([change == 3, change != 1], axis=1)
    for c, (s0, L) in enumerate(zip(cslot.tolist(), clen.tolist())):
        want = pair[s0:s0 + L][emit[s0:s0 + L]].tobytes().decode("ascii")
        assert got[c] == want, c


# ------------------------------------------------------------------------------------------------ public API
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["inf", "-inf", "nan", "1e19", "2.5"])
def test_public_api_min_depth_edges(golden, cases, name):
    """consensus_sequence and bam_to_consensus with min_depth values whose ceiling is no int64: the reference's
    answers (all N for inf and 1e19, never N for nan and -inf)."""
    md = dict(T.MIN_DEPTHS)[name]
    for seed in (1, 2, 3, 41):
        case = cases[seed]
        L, c = case["L"], case["counts"]
        weights = [{k: int(c[col, p]) for k, col in zip("ATGCN", (0, 3, 2, 1, 4))} for p in range(L)]
        insertions = [dict(case["insertions"].get(s, [])) for s in range(L + 1)]
        got = K.consensus_sequence(weights, insertions, c[5].tolist(), None, False, md, False)
        want = golden["cases"][str(seed)]["consensus"][name]
        assert [got[0], "".join("-" if x is None else x for x in got[1])] == want, seed
    root = os.path.dirname(GOLDEN)
    for rel, runs in golden["files"].items():
        path = os.path.join(root, rel)
        res = K.bam_to_consensus(path, min_depth=md)
        want = runs[name]
        assert [[r.name, r.sequence] for r in res.consensuses] == want["fasta"], rel
        assert {c: "".join("-" if x is None else x for x in ch) for c, ch in res.refs_changes.items()} == want["changes"]
        assert {c: rep.replace(path, "{path}") for c, rep in res.refs_reports.items()} == want["reports"], rel
