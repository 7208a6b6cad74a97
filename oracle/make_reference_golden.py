"""TEST INFRASTRUCTURE ONLY -- generates tests/golden/reference_runs.json.gz from the UNMODIFIED reference.

Run where a reference tree is present (see oracle/refload.py):   python -m oracle.make_reference_golden

It records what the reference returns on inputs the tests rebuild from seeds, so that the comparisons with
the reference run without it:
  fuzz        `parse_bam` on the 400 random alignments of tests/fuzz_cases.py: the exception raised, or per
              contig the sha256 of the int32 [19, L+1] table (tests/helpers.reference_alignment_to_table),
              the non-empty insertion dicts in first-seen order, and `changes` of `consensus_sequence`.
  host_api    for the clip-heavy alignments of tests/clip_cases.py (seeds 0..159) and the random ones
              (seeds 0..399), under the option sets of tests/test_fuzz_host_api.py: `bam_to_consensus`
              (FASTA, `changes`, reports with the input path replaced by "{path}") or its exception, the
              CDR helpers on the reference's own tables, and digests of the `weights` / `features` frames.
  fasta       the reference suite's own FASTA files (data fixtures; plain and --realign) keyed by the
              golden name of their input under tests/golden/inputs/.
  cuts        the first records of each of the 17 BAM/SAM fixtures of the reference suite, byte for byte
              (read names, qualities, aux tags as the aligners wrote them), stored as
              tests/golden/inputs/cut_<name>.bam / .sam, and `parse_bam` on them as for `fuzz`.
"""
from __future__ import annotations

import glob
import gzip
import json
import os
import struct
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import refload  # noqa: E402
from oracle.make_golden import FIXTURES  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "reference_runs.json.gz")
INPUTS = os.path.join(ROOT, "tests", "golden", "inputs")
CUT_RECORDS = {"mm2_gp120": 10, "ext_1_debug": 8, "ext_2_bc63": 8, "ext_3_bc75": 8}  # long reads; the others 60


def cut_fixture(src, dst_stem, n):
    """The header and the first n records of a BAM (raw record bytes, gzip) or SAM file; returns the new path."""
    if src.endswith(".sam"):
        lines = open(src).read().splitlines(True)
        body = [l for l in lines if l.startswith("@")] + [l for l in lines if not l.startswith("@")][:n]
        with open(dst_stem + ".sam", "wt") as fh:
            fh.write("".join(body))
        return dst_stem + ".sam"
    data = gzip.open(src, "rb").read()
    (l_text,) = struct.unpack_from("<i", data, 4)
    off = 8 + l_text
    (n_ref,) = struct.unpack_from("<i", data, off)
    off += 4
    for _ in range(n_ref):
        (l_name,) = struct.unpack_from("<i", data, off)
        off += 8 + l_name
    for _ in range(n):
        (block,) = struct.unpack_from("<i", data, off)
        off += 4 + block
    with gzip.GzipFile(dst_stem + ".bam", "wb", compresslevel=9, mtime=0) as fh:
        fh.write(data[:off])
    return dst_stem + ".bam"


def _raised(exc):
    return [type(exc).__name__] + ([exc.args[0]] if isinstance(exc, KeyError) else [])


def _regions(rs):
    return [list(r) for r in rs]


def fuzz_case(k, path):
    import helpers as H

    try:
        alns = k.parse_bam(path)
    except (IndexError, KeyError) as exc:
        return {"raises": _raised(exc)}
    out = {"contigs": list(alns), "table_sha256": [], "insertions": [], "changes": []}
    for aln in alns.values():
        t, ins = H.reference_alignment_to_table(aln)
        out["table_sha256"].append(H.table_sha256(t))
        out["insertions"].append([[i, list(d.items())] for i, d in enumerate(ins) if d])
        _, changes = k.consensus_sequence(aln.weights, aln.insertions, aln.deletions, None, False, 1, False)
        out["changes"].append(changes)
    return out


def host_api_case(k, path, seed, with_frames):
    import helpers as H
    import test_fuzz_host_api as T

    o = T._options(seed)
    args = [o[n] for n in T.OPTION_NAMES]
    case = {}
    try:
        res = k.bam_to_consensus(path, *args)
    except (IndexError, KeyError, ValueError) as exc:
        case["raises"] = type(exc).__name__
        return case
    case["fasta"] = [[r.name, r.sequence] for r in res.consensuses]
    case["changes"] = dict(res.refs_changes)
    case["reports"] = {c: rep.replace(path, "{path}") for c, rep in res.refs_reports.items()}
    case["cdr"] = []
    for aln in k.parse_bam(path).values():
        f = k.cdr_start_consensuses(aln.weights, aln.deletions, aln.clip_start_weights, aln.clip_start_depth,
                                    o["clip_decay_threshold"], o["mask_ends"])
        r = k.cdr_end_consensuses(aln.weights, aln.deletions, aln.clip_end_weights, aln.clip_end_depth,
                                  o["clip_decay_threshold"], o["mask_ends"])
        p = k.cdrp_consensuses(aln.weights, aln.deletions, aln.clip_start_weights, aln.clip_end_weights,
                               aln.clip_start_depth, aln.clip_end_depth, o["clip_decay_threshold"], o["mask_ends"])
        case["cdr"].append({"start": _regions(f), "end": _regions(r), "pairs": [[list(a), list(b)] for a, b in p],
                            "merged": _regions(k.merge_cdrps(p, o["min_overlap"]))})
    if with_frames:
        relative, confidence, alpha = T._frame_options(seed)
        case["weights_sha256"] = H.frame_sha256(k.weights(path, relative, confidence, alpha))
        try:
            case["features_sha256"] = H.frame_sha256(k.features(path))
        except IndexError:
            case["features_sha256"] = None
    return case


def reference_fasta():
    """{golden name: {"plain": {record: sequence}, "realign": {...}}} for every fixture that has FASTA files."""
    def read(path):
        recs, name = {}, None
        for line in open(path):
            line = line.strip()
            if line.startswith(">"):
                name = line[1:]
                recs[name] = ""
            elif name:
                recs[name] += line
        return recs

    out = {}
    for name, rel in FIXTURES:
        stem = os.path.splitext(os.path.join(refload.REFERENCE_ROOT, "tests", rel))[0]
        if os.path.isfile(stem + ".fa"):
            out[name] = {"plain": read(stem + ".fa"), "realign": read(stem + ".realign.fa")}
    return out


def main():
    import test_fuzz_host_api as T
    import test_fuzz_parity as P
    from clip_cases import clip_case
    from fuzz_cases import random_case

    if not refload.available() or not glob.glob(os.path.join(refload.REFERENCE_ROOT, "tests", "data_*")):
        raise SystemExit("no reference tree with its test data found; see oracle/refload.py")
    k = refload.load_reference()
    data = {"reference": "bede/kindel v1.2.1 @ 14d727b", "fuzz": [], "host_api": {"clip": [], "generic": []},
            "fasta": reference_fasta()}
    data["cuts"] = {}
    for name, rel in FIXTURES:
        path = cut_fixture(os.path.join(refload.REFERENCE_ROOT, "tests", rel), os.path.join(INPUTS, "cut_" + name),
                           CUT_RECORDS.get(name, 60))
        data["cuts"][name] = dict(fuzz_case(k, path), input=os.path.relpath(path, os.path.dirname(INPUTS)))
    with tempfile.TemporaryDirectory() as tmp:
        for seed in range(P.N_CASES):
            path = os.path.join(tmp, "fuzz%d.sam" % seed)
            with open(path, "wt") as fh:
                fh.write(random_case(seed))
            data["fuzz"].append(fuzz_case(k, path))
        for kind, n, make, every in (("clip", T.N_CLIP, clip_case, 4), ("generic", T.N_GENERIC, random_case, 3)):
            for seed in range(n):
                path = os.path.join(tmp, "%s%d.sam" % (kind, seed))
                with open(path, "wt") as fh:
                    fh.write(make(seed))
                data["host_api"][kind].append(host_api_case(k, path, seed, seed % every == 0))
    with gzip.GzipFile(OUT, "wb", mtime=0) as fh:
        fh.write(json.dumps(data, sort_keys=True, separators=(",", ":")).encode())
    print(OUT, os.path.getsize(OUT), "bytes")


if __name__ == "__main__":
    main()
