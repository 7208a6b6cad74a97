"""Differential fuzzing of the hot path on random small alignments (tests/fuzz_cases.py).

CPU (always):       C oracle == reference-shaped CPython port, including which exception is raised.
CPU (always):       C oracle == what the UNMODIFIED reference returned (tables, insertion dicts, changes, exceptions).
GPU (`-m gpu`):     engine through the public API == C oracle (tables, events, calls, exceptions)."""
import numpy as np
import pytest

import helpers as H
from fuzz_cases import random_case
from kindel_b200 import bamio
from oracle import coracle, py_oracle, samdecode

N_CASES = 400


def _load(tmp_path, seed):
    p = tmp_path / ("fuzz%d.sam" % seed)
    p.write_text(random_case(seed))
    return p


def _oracle_outcome(batch):
    try:
        counts, events = coracle.pileup(batch)
    except IndexError:
        return ("IndexError",), None, None
    except KeyError as exc:
        return ("KeyError", exc.args[0]), None, None
    return None, counts, events


def _py_outcome(path, batch):
    """py_oracle contig by contig, in the reference's order; first exception wins."""
    header, records = samdecode.read_alignment_file(path)
    lens = {sn[3:]: int(f[0][3:]) for sn, f in header["@SQ"].items()}
    groups = {}
    for r in records:
        groups.setdefault(r.rname, []).append(r)
    groups.pop("*", None)
    out = {}
    try:
        for name, recs in groups.items():
            out[name] = py_oracle.pileup(lens[name], [py_oracle.Rec(r.pos, r.mapped, r.seq, r.cigars) for r in recs])
    except IndexError:
        return ("IndexError",), None
    except KeyError as exc:
        return ("KeyError", exc.args[0].upper()), None
    return None, out


def test_c_oracle_vs_python_port(tmp_path):
    raised = 0
    for seed in range(N_CASES):
        path = _load(tmp_path, seed)
        try:
            batch = bamio.read_alignment(path)
        except ValueError:
            continue  # a base outside the BAM alphabet cannot be packed (documented deviation)
        err, counts, events = _oracle_outcome(batch)
        perr, tabs = _py_outcome(path, batch)
        assert err == perr, (seed, err, perr)
        if err:
            raised += 1
            continue
        assert list(tabs) == batch.contig_names, seed
        ins = H.events_to_dicts(batch, events)
        for c, (name, p) in enumerate(tabs.items()):
            t = H.contig_view(batch, counts, c)
            L = int(batch.contig_len[c])
            for k, b in enumerate("ACGTN"):
                assert [w[b] for w in p.weights] == t[k, :L].tolist(), (seed, name, b)
                assert [w[b] for w in p.clip_start_weights] == t[9 + k, :L].tolist(), (seed, "csw")
                assert [w[b] for w in p.clip_end_weights] == t[14 + k, :L].tolist(), (seed, "cew")
            assert p.deletions == t[5].tolist() and p.clip_starts == t[7].tolist() and p.clip_ends == t[8].tolist(), seed
            s0 = int(batch.contig_slot[c])
            for i, d in enumerate(p.insertions):
                assert list(d.items()) == list(ins.get(s0 + i, {}).items()), (seed, i)
            seq, changes = py_oracle.vote(p, 2)
            calls = coracle.vote(counts, 2)[s0:s0 + L]
            assert H.calls_to_changes(calls) == changes, seed
    assert raised > 20  # the generator really reaches the error paths


def test_c_oracle_vs_unmodified_reference(tmp_path):
    """The reference's outcome for every case (tests/golden/reference_runs.json.gz, oracle/make_reference_golden.py):
    the exception it raised, or its tables, insertion dicts in first-seen order and `changes`."""
    golden = H.reference_runs()["fuzz"]
    assert len(golden) == N_CASES
    raised = 0
    for seed in range(N_CASES):
        path = _load(tmp_path, seed)
        want = golden[seed]
        ref_err = tuple(want["raises"]) if "raises" in want else None
        try:
            batch = bamio.read_alignment(path)
        except ValueError:
            continue
        except KeyError:
            assert ref_err is not None and ref_err[0] == "KeyError"  # RNAME missing from @SQ
            continue
        err, counts, events = _oracle_outcome(batch)
        assert err == ref_err, (seed, err, ref_err)
        if err:
            raised += 1
            continue
        assert want["contigs"] == batch.contig_names
        ins = H.events_to_dicts(batch, events)
        calls = coracle.vote(counts, 1)
        for c in range(len(want["contigs"])):
            t = H.contig_view(batch, counts, c)
            assert H.table_sha256(t) == want["table_sha256"][c], seed
            s0, L = int(batch.contig_slot[c]), int(batch.contig_len[c])
            got_ins = [[i, [list(kv) for kv in ins[s0 + i].items()]] for i in range(L + 1) if ins.get(s0 + i)]
            assert got_ins == want["insertions"][c], seed
            assert H.calls_to_changes(calls[s0:s0 + L]) == want["changes"][c], seed
    assert raised > 20


@pytest.mark.gpu
def test_engine_vs_c_oracle(tmp_path):
    import torch

    from kindel_b200 import engine

    for seed in range(N_CASES):
        path = _load(tmp_path, seed)
        try:
            batch = bamio.read_alignment(path)
        except ValueError:
            continue
        err, counts, events = _oracle_outcome(batch)
        db = engine.upload(batch)
        if err:
            with pytest.raises({"IndexError": IndexError, "KeyError": KeyError}[err[0]]) as exc:
                engine.pileup(db)
            if err[0] == "KeyError":
                assert exc.value.args[0] == err[1], seed
            continue
        c, e = engine.pileup(db)
        torch.cuda.synchronize()
        np.testing.assert_array_equal(c.cpu().numpy(), counts, err_msg=str(seed))
        np.testing.assert_array_equal(e.cpu().numpy(), events, err_msg=str(seed))
        np.testing.assert_array_equal(engine.vote(c, 2).cpu().numpy(), coracle.vote(counts, 2), err_msg=str(seed))


def test_cpp_bam_decoder_equals_the_numpy_flatten_on_fuzz_cases(tmp_path):
    """The same random alignments as BAM through the C++ decoder (bam_host.cpp: filter, classification, inline CIGAR
    blocks, index lists, reach) and as SAM text through bamio.finalize (numpy): every array of the device layout must
    be identical, for several thread counts -- POS == 0, overhanging clips, exotic ops and bases, unmapped records and
    the other edge cases the generator makes included."""
    from oracle import samdecode as sd

    ops = "MIDNSHP=X"
    compared = 0
    for seed in range(0, N_CASES, 2):
        path = _load(tmp_path, seed)
        try:
            want = bamio.read_alignment(path)
        except ValueError:
            continue  # a base outside the BAM alphabet cannot be packed into 4 bits: no BAM of it exists either
        header, records = sd.read_alignment_file(path)
        names = [sn[3:] for sn in header["@SQ"]]
        contigs = [(nm, int(header["@SQ"]["SN:" + nm][0][3:])) for nm in names]
        recs = []
        for r in records:
            cig = [] if r.cigars == ((0, None),) else [(n << 4) | ops.index(o) for n, o in r.cigars]
            recs.append((names.index(r.rname) if r.rname != "*" else -1, r.pos - 1, r.flag, cig, r.seq.upper() if r.seq != "*" else "*"))
        bam = tmp_path / ("fuzz%d.bam" % seed)
        bamio.write_bam(bam, contigs, recs, level=1)
        for threads in (1, 5):
            got = bamio.read_bam(bam, threads=threads)
            assert got.contig_names == want.contig_names and got.n_records == want.n_records, seed
            for f in ("contig_len", "contig_read_off", "contig_slot", "ref_start", "seq_len", "l_seq", "seq_off", "seq4",
                      "cig_off", "cigar", "complex_idx", "hard_idx"):
                np.testing.assert_array_equal(getattr(got, f), getattr(want, f), err_msg="seed %d %s" % (seed, f))
            assert (got.n_events, got.reads_sorted, got.max_simple_len, got.reach_right, got.reach_left, got.aligned_bases) == \
                   (want.n_events, want.reads_sorted, want.max_simple_len, want.reach_right, want.reach_left, want.aligned_bases), seed
        compared += 1
    assert compared > 100
