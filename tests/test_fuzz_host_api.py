"""Differential fuzzing of the HOST halves of the API against what the unmodified reference returned.

For random clip-heavy alignments (tests/clip_cases.py) and the generic fuzz cases (tests/fuzz_cases.py):
`bam_to_consensus` under random option sets (realign on/off, min_depth, min_overlap, clip_decay_threshold,
mask_ends, trim_ends, uppercase) -- sequences, changes and report text -- the CDR helper functions called
the way the reference's tests call them, and the `weights` / `features` frames.  Count tables come from the
CPU oracle (`PileupRun.from_host_tables`), so the code under test is exactly the host code the GPU engine
feeds; no GPU is needed.  The reference's results for the same seeds and options are stored in
tests/golden/reference_runs.json.gz (oracle/make_reference_golden.py)."""
import random

import pytest

import helpers as H
from clip_cases import clip_case
from fuzz_cases import random_case
from kindel_b200 import bamio
from kindel_b200 import kindel as K
from oracle import coracle

N_CLIP = 160
N_GENERIC = 400  # most generic cases abort in the pileup (by design); the survivors are tiny odd contigs
OPTION_NAMES = ("realign", "min_depth", "min_overlap", "clip_decay_threshold", "mask_ends", "trim_ends", "uppercase")
_ERRORS = {"IndexError": IndexError, "KeyError": KeyError, "ValueError": ValueError}


def _run(path):
    batch = bamio.read_alignment(path)
    counts, events = coracle.pileup(batch)
    return K.PileupRun.from_host_tables(batch, counts, coracle.derive(counts), events), counts


def _options(seed):
    rng = random.Random(seed)
    return dict(realign=rng.random() < 0.8, min_depth=rng.choice([1, 1, 2, 5]), min_overlap=rng.choice([1, 3, 7, 9]),
                clip_decay_threshold=rng.choice([0.0, 0.1, 0.1, 0.3, 0.9]), mask_ends=rng.choice([0, 1, 5, 20, 50]),
                trim_ends=rng.random() < 0.5, uppercase=rng.random() < 0.3)


def _frame_options(seed):
    """(relative, confidence, alpha) of the `weights` frame compared for a seed."""
    rng = random.Random(seed)
    return rng.random() < 0.5, rng.random() < 0.7, rng.choice([0.01, 0.05, 0.2])


def _regions(rs):
    return [list(r) for r in rs]


def _compare_consensus(want, path, seed, stats):
    o = _options(seed)
    args = [o[n] for n in OPTION_NAMES]
    try:
        run, counts = _run(path)
    except (IndexError, KeyError, ValueError) as exc:
        assert "raises" in want, (seed, exc)
        return None, None
    if "raises" in want:
        # the pileup succeeded on our side, so the reference failed later (host logic): same exception here
        with pytest.raises(_ERRORS[want["raises"]]):
            K.consensus_from_run(run, coracle.vote(counts, o["min_depth"]), str(path), *args)
        stats["raised"] += 1
        return None, None
    got = K.consensus_from_run(run, coracle.vote(counts, o["min_depth"]), str(path), *args)
    assert [[r.name, r.sequence] for r in got.consensuses] == want["fasta"], (seed, o)
    assert dict(got.refs_changes) == want["changes"], (seed, o)
    assert {c: rep.replace(str(path), "{path}") for c, rep in got.refs_reports.items()} == want["reports"], (seed, o)
    if o["realign"]:
        for rep in want["reports"].values():  # reports that list at least one merged clip-dominant region
            line = next(l for l in rep.splitlines() if l.startswith("- clip-dominant regions"))
            stats["patched"] += line.strip() != "- clip-dominant regions:"
    return run, counts


def _compare_cdr_functions(want, run, counts, seed, stats):
    """cdr_start / cdr_end / cdrp_consensuses / merge_cdrps on the reference's list-of-dict tables (rebuilt from
    the oracle's table) and on the engine's views must give the reference's Regions."""
    o = _options(seed)
    thr, mask = o["clip_decay_threshold"], o["mask_ends"]
    batch = run.batch
    assert len(want) == len(batch.contig_names), seed
    for c, (name, w) in enumerate(zip(batch.contig_names, want)):
        weights, dels, csw, cew, csd, ced = H.reference_lists(H.contig_view(batch, counts, c), int(batch.contig_len[c]))
        mine = run.alignment(c)
        assert _regions(K.cdr_start_consensuses(weights, dels, csw, csd, thr, mask)) == w["start"], (seed, name, "fwd/lists")
        assert _regions(K.cdr_start_consensuses(mine.weights, mine.deletions, mine.clip_start_weights,
                                                mine.clip_start_depth, thr, mask)) == w["start"], (seed, name, "fwd/views")
        assert _regions(K.cdr_end_consensuses(weights, dels, cew, ced, thr, mask)) == w["end"], (seed, name, "rev/lists")
        assert _regions(K.cdr_end_consensuses(mine.weights, mine.deletions, mine.clip_end_weights,
                                              mine.clip_end_depth, thr, mask)) == w["end"], (seed, name, "rev/views")
        got_p = K.cdrp_consensuses(weights, dels, csw, cew, csd, ced, thr, mask)
        assert [[list(f), list(r)] for f, r in got_p] == w["pairs"], (seed, name)
        assert _regions(K.merge_cdrps(got_p, o["min_overlap"])) == w["merged"], (seed, name)
        stats["regions"] += len(w["start"]) + len(w["end"])
        stats["pairs"] += len(w["pairs"])


def _compare_frames(want, run, seed):
    relative, confidence, alpha = _frame_options(seed)
    assert H.frame_sha256(K.weights_from_run(run, relative, confidence, alpha)) == want["weights_sha256"], seed
    if want["features_sha256"] is None:
        with pytest.raises(IndexError):
            K.features_from_run(run)
        return
    assert H.frame_sha256(K.features_from_run(run)) == want["features_sha256"], seed


def test_clip_heavy_cases_against_reference(tmp_path):
    golden = H.reference_runs()["host_api"]["clip"]
    assert len(golden) == N_CLIP
    stats = dict(raised=0, patched=0, regions=0, pairs=0)
    for seed in range(N_CLIP):
        path = tmp_path / ("clip%d.sam" % seed)
        path.write_text(clip_case(seed))
        want = golden[seed]
        run, counts = _compare_consensus(want, path, seed, stats)
        if run is None:
            continue
        _compare_cdr_functions(want["cdr"], run, counts, seed, stats)
        if seed % 4 == 0:
            _compare_frames(want, run, seed)
    # the generator really reaches the realign machinery
    assert stats["regions"] > 100 and stats["pairs"] > 20 and stats["patched"] > 10, stats


def test_generic_cases_host_api_against_reference(tmp_path):
    golden = H.reference_runs()["host_api"]["generic"]
    assert len(golden) == N_GENERIC
    stats = dict(raised=0, patched=0, regions=0, pairs=0)
    done = 0
    for seed in range(N_GENERIC):
        path = tmp_path / ("gen%d.sam" % seed)
        path.write_text(random_case(seed))
        want = golden[seed]
        if want.get("raises") == "ValueError":
            continue  # a base outside the BAM alphabet cannot be packed (documented deviation)
        run, counts = _compare_consensus(want, path, seed, stats)
        if run is None:
            continue
        done += 1
        _compare_cdr_functions(want["cdr"], run, counts, seed, stats)
        if seed % 3 == 0:
            _compare_frames(want, run, seed)
    assert done > 20
