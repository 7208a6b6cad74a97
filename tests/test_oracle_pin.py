"""Pins the oracle: the C restatement (oracle/kindel_oracle.c) against
  (a) the golden vectors the UNMODIFIED reference produced (tests/golden/, oracle/make_golden.py), and
  (b) the reference's known-answer integers of its tests/test_kindel.py:63-89 and the FASTA files of its
      own test-suite (tests/golden/reference_runs.json.gz).
No GPU involved."""
import os
from collections import OrderedDict

import numpy as np
import pytest

import helpers as H
from conftest import GOLDEN, golden_input
from kindel_b200 import bamio
from oracle import coracle, samdecode


def test_golden_tables_insertions_and_vote(manifest, golden_npz):
    for name, entry in manifest["files"].items():
        batch = bamio.read_alignment(golden_input(entry))
        counts, events = coracle.pileup(batch)
        derived = coracle.derive(counts)
        ins = H.events_to_dicts(batch, events)
        g = golden_npz(name)
        assert batch.contig_names == [c["name"] for c in entry["contigs"]]
        calls = coracle.vote(counts, 1)
        for c, meta in enumerate(entry["contigs"]):
            L = meta["ref_len"]
            s0 = int(batch.contig_slot[c])
            assert int(batch.contig_len[c]) == L
            np.testing.assert_array_equal(H.contig_view(batch, counts, c), g["c%d_counts" % c], err_msg=name)
            np.testing.assert_array_equal(derived[0, s0:s0 + L], g["c%d_consensus_depth" % c])
            np.testing.assert_array_equal(derived[1, s0:s0 + L], g["c%d_clip_start_depth" % c])
            np.testing.assert_array_equal(derived[2, s0:s0 + L], g["c%d_clip_end_depth" % c])
            np.testing.assert_array_equal(derived[3, s0:s0 + L], g["c%d_clip_depth" % c])
            want = {s0 + i: [tuple(kv) for kv in items] for i, items in meta["insertions"]}
            got = {s: list(d.items()) for s, d in ins.items() if s0 <= s <= s0 + L}
            assert got == want, name
            changes = "".join("-" if c_ is None else c_ for c_ in H.calls_to_changes(calls[s0:s0 + L]))
            assert changes == entry["runs"]["plain"]["changes"][meta["name"]], name


def _case_batch(case, tmp_path):
    p = tmp_path / (case["name"] + ".sam")
    p.write_text(case["sam"])
    return bamio.read_alignment(p), p


def test_edge_cases_match_the_reference(manifest, tmp_path):
    """SURVEY.md Appendix A behaviours, each pinned by the reference's own output."""
    assert len(manifest["edge_cases"]) >= 40
    for case in manifest["edge_cases"]:
        batch, _ = _case_batch(case, tmp_path)
        if case["raises"]:
            kind, args = case["raises"]
            with pytest.raises({"IndexError": IndexError, "KeyError": KeyError}[kind]) as exc:
                coracle.pileup(batch)
            if kind == "KeyError":
                assert [str(a) for a in exc.value.args] == args, case["name"]
            continue
        counts, events = coracle.pileup(batch)
        assert batch.contig_names == case["contigs"]
        np.testing.assert_array_equal(H.contig_view(batch, counts, 0), np.array(case["counts"]), err_msg=case["name"])
        got = {s: list(d.items()) for s, d in H.events_to_dicts(batch, events).items()}
        assert got == {i: [tuple(kv) for kv in items] for i, items in case["insertions"]}, case["name"]
        L = int(batch.contig_len[0])
        for md in (1, 3):
            calls = coracle.vote(counts, md)[:L]
            changes = "".join("-" if c is None else c for c in H.calls_to_changes(calls))
            assert changes == case["changes_min_depth_%d" % md], case["name"]


def test_oracle_decoder_and_product_decoder_agree(manifest):
    """Two independent BAM/SAM decoders (stdlib struct vs C++ gather) see the same records."""
    for name, entry in manifest["files"].items():
        path = golden_input(entry)
        _, records = samdecode.read_alignment_file(path)
        batch = bamio.read_alignment(path)
        kept = [r for r in records if r.mapped and len(r.seq) > 1 and r.rname != "*"]
        assert batch.n_records == len(records)
        assert batch.n_reads == len(kept)
        order = OrderedDict()
        for r in records:
            if r.rname != "*":
                order.setdefault(r.rname, []).append(r)
        assert list(order) == batch.contig_names
        flat = [r for rs in order.values() for r in rs if r.mapped and len(r.seq) > 1]
        for k in list(range(0, len(flat), max(1, len(flat) // 200))):
            r = flat[k]
            assert int(batch.ref_start[k]) == r.pos - 1
            words = batch.cigar[int(batch.cig_off[k]):int(batch.cig_off[k + 1])].tolist()
            assert [(w >> 4, "MIDNSHP=X"[w & 15]) for w in words] == [c for c in r.cigars if c[1] is not None]
            assert H.event_string(batch, k, 0, len(r.seq)) == r.seq.upper() or int(batch.l_seq[k]) >= 0


def test_reference_known_answers(golden_npz, manifest):
    """reference tests/test_kindel.py:63-89: the known-answer integers, in the reference's own tables (tests/golden/)
    and in the C oracle's tables of the same inputs."""
    def tables(name):
        batch = bamio.read_alignment(golden_input(manifest["files"][name]))
        counts, _ = coracle.pileup(batch)
        assert len(batch.contig_names) == 1
        return batch, [golden_npz(name)["c0_counts"], H.contig_view(batch, counts, 0)]

    batch, t1 = tables("bwa_1_1")
    batch2, t2 = tables("ext_3_bc75")
    assert batch.contig_names == ["ENA|EU155341|EU155341.2"] and int(batch.contig_len[0]) == 9306
    for t, t_2 in zip(t1, t2):
        A, G, T, DEL, INS, CLIP_S, CLIP_E = 0, 2, 3, 5, 6, 7, 8
        assert t.shape[1] == 9307
        assert t[A, 0] == 22 and t[A, 23] == 57
        assert t_2[G, 68] == 1 and t_2[T, 2368] == 13
        assert [t_2[DEL, i] for i in (399, 402, 411, 1048, 1049, 1050)] == [14, 14, 15, 14, 14, 14]
        assert t_2[CLIP_E, 1748] == 12
        assert t[CLIP_S, 525] == 16 and t[CLIP_S, 1437] == 84
        assert t_2[INS, 453] == 14 and t_2[INS, 457] == 14


def test_c_oracle_equals_reference_on_every_reference_fixture():
    """The first records of all 17 BAM/SAM fixtures of the reference's test-suite, byte for byte as the aligners
    wrote them (read names, qualities, aux tags; tests/golden/inputs/cut_*), through the product decoder and the C
    oracle == what the reference returned for them (oracle/make_reference_golden.py): tables, insertion dicts with
    their first-seen order, and the vote."""
    cuts = H.reference_runs()["cuts"]
    assert len(cuts) == 17
    for name, want in cuts.items():
        assert "raises" not in want, name
        batch = bamio.read_alignment(os.path.join(GOLDEN, want["input"]))
        counts, events = coracle.pileup(batch)
        calls = coracle.vote(counts, 1)
        ins = H.events_to_dicts(batch, events)
        assert batch.contig_names == want["contigs"], name
        for c in range(len(want["contigs"])):
            assert H.table_sha256(H.contig_view(batch, counts, c)) == want["table_sha256"][c], name
            s0, L = int(batch.contig_slot[c]), int(batch.contig_len[c])
            got_ins = [[i, [list(kv) for kv in ins[s0 + i].items()]] for i in range(L + 1) if ins.get(s0 + i)]
            assert got_ins == want["insertions"][c], name
            assert H.calls_to_changes(calls[s0:s0 + L]) == want["changes"][c], name


def test_golden_fasta_files_of_the_reference_suite(manifest):
    """The reference's own golden FASTA files (plain + realign; tests/golden/reference_runs.json.gz) against oracle
    tables + host code: 21 of 22, the 22nd belongs to a test the reference has commented out
    (tests/test_kindel.py:281-299) and the reference itself does not reproduce it."""
    from kindel_b200 import kindel as K

    fasta = H.reference_runs()["fasta"]
    assert len(fasta) == 11
    ok, bad = 0, []
    for name, want in sorted(fasta.items()):
        path = golden_input(manifest["files"][name])
        batch = bamio.read_alignment(path)
        counts, events = coracle.pileup(batch)
        run = K.PileupRun.from_host_tables(batch, counts, coracle.derive(counts), events)
        for realign in (False, True):
            kind = "realign" if realign else "plain"
            res = K.consensus_from_run(run, coracle.vote(counts, 1), path, realign, 1, 7, 0.1, 50, False, False)
            if {r.name: r.sequence for r in res.consensuses} == want[kind]:
                ok += 1
            else:
                bad.append((name, kind))
    assert ok == 21 and bad == [("ext_3_bc75", "realign")]


def test_python_port_against_golden(manifest, golden_npz):
    """oracle/py_oracle.py (the reference-shaped CPython loop timed by `bench.py --impl reference`)
    reproduces the reference's tables, insertion dicts and consensus on the small golden files."""
    from oracle import py_oracle

    for name in ("mm2_multi", "ext_3_bc75", "mm2_gp120"):
        entry = manifest["files"][name]
        header, records = samdecode.read_alignment_file(golden_input(entry))
        lens = {sn[3:]: int(next(f for f in fields if f.startswith("LN:"))[3:]) for sn, fields in header["@SQ"].items()}
        groups = OrderedDict()
        for r in records:
            if r.rname != "*":
                groups.setdefault(r.rname, []).append(py_oracle.Rec(r.pos, r.mapped, r.seq, r.cigars))
        g = golden_npz(name)
        assert list(groups) == [c["name"] for c in entry["contigs"]]
        for c, (ctg, recs) in enumerate(groups.items()):
            p = py_oracle.pileup(lens[ctg], recs)
            t = g["c%d_counts" % c]
            L = lens[ctg]
            for k, b in enumerate("ACGTN"):
                assert [w[b] for w in p.weights] == t[k, :L].tolist()
                assert [w[b] for w in p.clip_start_weights] == t[9 + k, :L].tolist()
                assert [w[b] for w in p.clip_end_weights] == t[14 + k, :L].tolist()
            assert p.deletions == t[5].tolist() and p.clip_starts == t[7].tolist() and p.clip_ends == t[8].tolist()
            assert list(p.consensus_depth) == g["c%d_consensus_depth" % c].tolist()
            want_ins = {i: [tuple(kv) for kv in items] for i, items in entry["contigs"][c]["insertions"]}
            assert {i: list(d.items()) for i, d in enumerate(p.insertions) if d} == want_ins
            seq, changes = py_oracle.vote(p, 1)
            assert seq == dict(map(tuple, entry["runs"]["plain"]["fasta"]))[ctg + "_cns"]
            assert "".join("-" if c_ is None else c_ for c_ in changes) == entry["runs"]["plain"]["changes"][ctg]


def _digest_check(table_i32, seq, changes, meta):
    import hashlib

    assert hashlib.sha256(np.ascontiguousarray(table_i32, dtype=np.int32).tobytes()).hexdigest() == meta["table_sha256"]
    assert [int(x) for x in table_i32.sum(axis=1)] == meta["column_sums"]
    assert len(seq) == meta["fasta_len"] and hashlib.sha256(seq.encode()).hexdigest() == meta["fasta_sha256"]
    assert hashlib.sha256("".join("-" if c is None else c for c in changes).encode()).hexdigest() == meta["changes_sha256"]


def test_megabase_fixture_digest(manifest):
    """The 6.1 Mb fixture of the reference (`bact.tiny`, secondary alignments with SEQ `*`, 8x depth):
    the oracle's dense table, consensus and changes hash to what the reference produced."""
    from kindel_b200 import kindel as K

    for name, entry in manifest["digests"].items():
        batch = bamio.read_alignment(golden_input(entry))
        counts, events = coracle.pileup(batch)
        calls = coracle.vote(counts, 1)
        ins = H.events_to_dicts(batch, events)
        assert batch.contig_names == [c["name"] for c in entry["contigs"]]
        for c, meta in enumerate(entry["contigs"]):
            s0, L = int(batch.contig_slot[c]), meta["ref_len"]
            want_ins = {s0 + i: [tuple(kv) for kv in items] for i, items in meta["insertions"]}
            assert {s: list(d.items()) for s, d in ins.items()} == want_ins
            seq, changes = K.assemble_consensus(calls[s0:s0 + L],
                                                lambda p: K.dict_consensus(ins.get(s0 + p, {})))
            _digest_check(H.contig_view(batch, counts, c), seq, changes, meta)
