"""K0 + the tile-owner kernel K1 (and every other kernel), SOURCE-level, on the CPU.

tests/emu/ compiles kindel_b200/csrc/*.cu for the host and runs the kernels under a functional model of the CUDA
execution model (tests/emu/cuda_emu.h); the tables must equal the C oracle's.  This checks what a numpy model of
the arithmetic (tests/k1f_model.py) cannot: the kernel's own indexing, sentinels, item splitting, flush conditions,
coverage scan, store / add / atomic modes, the depth split, the explosion of complex reads into pieces and sparse
updates, and the staging protocol (full / landed / empty mbarriers, producer barrier, cp.async prefetch).
It does not model timing or the memory model; the `-m gpu` parity tests remain the proof on the device."""
import numpy as np
import pytest

import emu_harness as E
from kindel_b200 import distributed as D
from kindel_b200 import synth
from oracle import coracle

pytestmark = pytest.mark.skipif(not E.available(), reason="needs g++ and the CUDA headers")

CASES = {
    "shallow":      lambda: synth.simple_reads(5, [3000], 40),
    "deep":         lambda: synth.simple_reads(71, [2000], 3000),            # > 31 blocks per window: mid-window flushes
    "long_reads":   lambda: synth.simple_reads(73, [9000], 600, read_len=6000),  # staging capacity splits sub-chunks
    "sparse":       lambda: synth.simple_reads(74, [50_000], 0.5),           # mostly empty tiles and windows
    "multi_contig": lambda: synth.simple_reads(75, [151, 200, 9000, 333, 160, 700], 40),  # several contigs per tile
    "len_1203":     lambda: synth.simple_reads(76, [20_000], 40, read_len=1203),
    "cfg4_like":    lambda: synth.simple_reads(77, [60_000], 200),
    "short_reads":  lambda: synth.simple_reads(78, [5000], 60, read_len=9),
}


@pytest.mark.parametrize("cx", [False, True], ids=["lean", "cx"])
@pytest.mark.parametrize("name", list(CASES))
def test_tile_owner_kernel_source_equals_oracle(name, cx):
    """Simple reads through both instantiations of K1 (the kCx one has smaller stages and the piece machinery)."""
    batch = CASES[name]()
    want, _ = coracle.pileup(batch)
    for mode in (E.F_ADD, E.F_STORE):
        got = E.run_pileup(batch, mode, cx=cx)
        np.testing.assert_array_equal(got[:5], want[:5], err_msg="%s mode=%s" % (name, mode))
        assert not got[5:].any()


@pytest.mark.parametrize("split", [2, 5])
@pytest.mark.parametrize("name", ["deep", "cfg4_like", "multi_contig", "sparse"])
def test_depth_split_units_share_a_tile(name, split):
    """`split` CTAs per tile, each a contiguous part of the tile's reads, flushing with REDs into a zeroed table."""
    batch = CASES[name]()
    want, _ = coracle.pileup(batch)
    got = E.run_pileup(batch, E.F_ATOMIC, split=split, grid=7)
    np.testing.assert_array_equal(got[:5], want[:5])
    assert not got[5:].any()


CX_CASES = {
    "cfg3_like":    lambda: synth.complex_reads(72, 6000, 60),                  # clips + indels + edge tail (hard reads)
    "cfg3_deep":    lambda: synth.complex_reads(91, 1500, 900, edge_tail=False),  # piece list overflows: items are cut
    "long_complex": lambda: synth.complex_reads(92, 9000, 30, read_len=900, edge_tail=False),
}


@pytest.mark.parametrize("name", list(CX_CASES) + ["mixed"])
def test_rare_complex_reads_by_atomics(name):
    """The other way kdl_pileup_range handles tile-eligible complex reads (when they are rare): the lean K1 treats them
    as inert and K1e counts their M/=/X bases too, with REDs behind the tile stores."""
    batch = synth.mixed_reads(93, [9000, 4000], 80, 0.05) if name == "mixed" else CX_CASES[name]()
    want_c, want_e = coracle.pileup(batch)
    hard = D.select_reads(batch, batch.hard_idx)
    wh = coracle.pileup(hard)[0] if batch.n_hard else 0
    for mode in (E.F_ADD, E.F_STORE):
        got, ev = E.run_pileup(batch, mode, cx=False, want_events=True, zero_rest=mode == E.F_STORE)
        np.testing.assert_array_equal(got, want_c - wh)


@pytest.mark.parametrize("split", [1, 3])
@pytest.mark.parametrize("name", list(CX_CASES))
def test_complex_reads_in_the_tile_kernel(name, split):
    """Tile-eligible complex reads: M segments as masked pieces through the bit-sliced counters, I / D / clip
    updates and insertion events from the producers; hard reads (K1g) on top."""
    batch = CX_CASES[name]()
    assert batch.n_complex > batch.n_hard
    want_c, want_e = coracle.pileup(batch)
    got_c, got_e = E.pileup_pipeline(batch, split=split)
    np.testing.assert_array_equal(got_c, want_c)
    np.testing.assert_array_equal(got_e, want_e)
    if split == 1:  # stale columns are overwritten / zeroed in the flush, K1 + K1e = everything but the hard reads
        got2, ev2 = E.run_pileup(batch, E.F_STORE, want_events=True, zero_rest=True)
        hard = __import__("kindel_b200.distributed", fromlist=["x"]).select_reads(batch, batch.hard_idx)
        wh, _ = coracle.pileup(hard)
        np.testing.assert_array_equal(got2, want_c - wh)


@pytest.mark.parametrize("mode", [E.F_ADD, E.F_STORE], ids=["add", "store"])
def test_accumulate_and_slot_ranges(mode):
    """Two batches added into one table (accumulate mode), then a fresh pass over a tile sub-range only."""
    a = synth.simple_reads(81, [20_000], 30)
    b = synth.simple_reads(81, [20_000], 50, read_seed=9)
    wa, _ = coracle.pileup(a)
    wb, _ = coracle.pileup(b)
    t = E.run_pileup(a, E.F_ADD)
    t = E.run_pileup(b, E.F_ADD, counts=t)
    np.testing.assert_array_equal(t[:5], (wa + wb)[:5])
    # overwrite (F_STORE) / add (F_ADD) on tiles [7, 19) with batch a: outside the range untouched
    lo, n = 7, 12
    t2 = E.run_pileup(a, mode, tile_lo=lo, n_tiles=n, counts=t.copy())
    s0, s1 = lo * 512, (lo + n) * 512
    inside = wa[:5, s0:s1] if mode == E.F_STORE else (t + wa)[:5, s0:s1]
    np.testing.assert_array_equal(t2[:5, s0:s1], inside)
    np.testing.assert_array_equal(t2[:5, :s0], t[:5, :s0])
    np.testing.assert_array_equal(t2[:5, s1:], t[:5, s1:])


def test_emulator_catches_a_staging_bug():
    """The emulator is not vacuous: a kernel that skips the wait for its bulk copy reads garbage here."""
    lib = E.load()
    assert lib.emu_selftest_missing_wait() == 1   # data read before mbar_wait differs from the source
    assert lib.emu_selftest_missing_wait_fixed() == 0


# ---- the rest of the kernels: K1s, K1g, diagnose, K2 (vote), derive, K2p (peer vote) ------------------------
def _oracle_outcome(batch):
    try:
        return None, coracle.pileup(batch)
    except IndexError:
        return ("IndexError",), None
    except KeyError as exc:
        return ("KeyError", exc.args[0]), None


def test_whole_pipeline_on_the_fuzz_cases(tmp_path):
    """Every kernel kdl_pileup / kdl_vote / kdl_derive / kdl_diagnose launches, source-level, on the 400 random
    alignments of tests/fuzz_cases.py: tables, insertion events, calls, derived columns and the exception
    (type and KeyError argument) equal the oracle's."""
    from fuzz_cases import random_case

    from kindel_b200 import bamio

    raised = done = 0
    for seed in range(400):
        path = tmp_path / ("fuzz%d.sam" % seed)
        path.write_text(random_case(seed))
        try:
            batch = bamio.read_alignment(path)
        except (ValueError, KeyError):
            continue
        err, res = _oracle_outcome(batch)
        if err:
            raised += 1
            with pytest.raises({"IndexError": IndexError, "KeyError": KeyError}[err[0]]) as exc:
                E.pileup_pipeline(batch)
            if err[0] == "KeyError":
                assert exc.value.args[0] == err[1], seed
            continue
        counts, events = res
        got_c, got_e = E.pileup_pipeline(batch)
        np.testing.assert_array_equal(got_c, counts, err_msg=str(seed))
        np.testing.assert_array_equal(got_e, events, err_msg=str(seed))
        if seed % 4 == 0:
            np.testing.assert_array_equal(E.vote(got_c, 2), coracle.vote(counts, 2), err_msg=str(seed))
            np.testing.assert_array_equal(E.derive(got_c), coracle.derive(counts), err_msg=str(seed))
        done += 1
    assert raised > 20 and done > 20


def test_mixed_batch_pipeline():
    """Config-3 shape (clips, indels, edge-case tail; most reads complex, some simple) end to end: K1 + K1g into one
    table, then the vote and the derived columns."""
    batch = synth.complex_reads(72, 6000, 60)
    want_c, want_e = coracle.pileup(batch)
    got_c, got_e = E.pileup_pipeline(batch)
    np.testing.assert_array_equal(got_c, want_c)
    np.testing.assert_array_equal(got_e, want_e)
    np.testing.assert_array_equal(E.vote(got_c, 1), coracle.vote(want_c, 1))
    np.testing.assert_array_equal(E.vote(got_c, 7), coracle.vote(want_c, 7))
    np.testing.assert_array_equal(E.derive(got_c), coracle.derive(want_c))


def test_unsorted_batches_take_the_atomic_kernels():
    batch = synth.complex_reads(72, 6000, 20)
    from kindel_b200 import distributed as D

    perm = np.random.default_rng(3).permutation(batch.n_reads)
    shuffled = D.select_reads(batch, perm)
    assert not shuffled.reads_sorted and not E.tileable(shuffled)
    want_c, want_e = coracle.pileup(shuffled)
    got_c, got_e = E.pileup_pipeline(shuffled)
    np.testing.assert_array_equal(got_c, want_c)
    np.testing.assert_array_equal(got_e, want_e)


def test_peer_vote_over_footprints():
    """K2p: the vote of the sum of per-rank tables, each read only inside its footprint, on an owner slice."""
    from kindel_b200 import distributed as D

    batch = synth.complex_reads(73, 5000, 40)
    full, _ = coracle.pileup(batch)
    shards = [D.shard_batch(batch, r, 3) for r in range(3)]
    tables = [coracle.pileup(s)[0] for s in shards]
    feet = [D.footprint(s) for s in shards]
    np.testing.assert_array_equal(sum(tables), full)
    want = coracle.vote(full, 2)
    n_slots = full.shape[1]
    for lo, hi in D.owner_slices(n_slots, 3):
        calls, reduced = E.vote_peers(tables, feet, lo, hi, 2, want_reduced=True)
        np.testing.assert_array_equal(calls[lo:hi], want[lo:hi])
        np.testing.assert_array_equal(reduced[:, lo:hi], full[:7, lo:hi])


@pytest.mark.parametrize("cut", ["equal", "footprint", "contigs"])
@pytest.mark.parametrize("world", [2, 3])
def test_fused_exchange_epochs(world, cut):
    """K2x + K2g for all ranks of a sharded pileup, three epochs with different data (flags compare epochs), the
    tables and call buffers alternating by epoch parity as distributed.ShardedConsensus does: every rank ends up
    with the complete call bytes of the summed table.  Slices cut equally, along the footprints (the core of a
    slice then reads no peer), or along whole contigs (no shared slot at all)."""
    from kindel_b200 import distributed as D

    flags = {k: [np.zeros(16, dtype=np.int32) for _ in range(world)] for k in ("ready", "done")}
    flags["counter"] = [np.zeros(1, dtype=np.int32) for _ in range(world)]
    bufs = None
    for epoch, seed in ((1, 74), (2, 75), (3, 76)):
        if cut == "contigs":
            batch = synth.simple_reads(seed, [1800, 2500, 700, 1900], 25)
            shards = [D.shard_by_contig(batch, r, world) for r in range(world)]
        else:
            batch = synth.complex_reads(seed, 7000, 30)
            shards = [D.shard_batch(batch, r, world) for r in range(world)]
        full, _ = coracle.pileup(batch)
        tables = [coracle.pileup(s)[0] for s in shards]
        feet = [D.footprint(s) for s in shards]
        n_slots = full.shape[1]
        slices = D.owner_slices(n_slots, world) if cut == "equal" else D.footprint_slices(feet, n_slots)
        if bufs is None:
            bufs = [[np.full(n_slots, 0xEE, dtype=np.uint8) for _ in range(world)] for _ in range(2)]
        calls = bufs[epoch & 1]
        E.exchange_epoch(tables, feet, slices, calls, flags, epoch, min_depth=2)
        want = coracle.vote(full, 2)
        for r in range(world):
            np.testing.assert_array_equal(calls[r], want, err_msg="epoch %d rank %d" % (epoch, r))
            assert (flags["ready"][r][:world] == epoch).all() and (flags["done"][r][:world] == epoch).all()


@pytest.mark.parametrize("schedule,seed", [("reverse", 0), ("random", 1), ("random", 2)])
def test_other_thread_interleavings(schedule, seed):
    """The staging protocol (full / landed / empty mbarrier ring, producer barrier, cp.async prefetch, the piece
    queue of the consumers) under other thread orders than the emulator's default."""
    E.set_schedule(schedule, seed)
    try:
        for name in ("shallow", "multi_contig", "long_reads"):
            batch = CASES[name]()
            want, _ = coracle.pileup(batch)
            got = E.run_pileup(batch, E.F_STORE, grid=4)
            np.testing.assert_array_equal(got[:5], want[:5], err_msg="%s %s/%d" % (name, schedule, seed))
        batch = CX_CASES["cfg3_like"]()
        want_c, want_e = coracle.pileup(batch)
        got_c, got_e = E.pileup_pipeline(batch)
        np.testing.assert_array_equal(got_c, want_c)
        np.testing.assert_array_equal(got_e, want_e)
    finally:
        E.set_schedule("forward")
