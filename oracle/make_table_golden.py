"""TEST INFRASTRUCTURE ONLY -- generates tests/golden/table_runs.json.gz from the UNMODIFIED reference.

Run where a reference tree is present (see oracle/refload.py):   python -m oracle.make_table_golden

It feeds the adversarial count tables of tests/table_cases.py straight into the reference's per-position
functions, built as the reference builds its own inputs (parse_records, kindel/kindel.py:29-39): `weights` and the
clip weights as lists of dicts in A,T,G,C,N order, `deletions` and `insertions` of length L + 1, every insertion dict
in first-seen order, and the clip depths as the ACGT sums (kindel.py:90-95).  Per case seed it stores only what the
reference returned:
  consensus   `consensus_sequence(...)` -> [sequence, changes] for every min_depth of table_cases.MIN_DEPTHS
              (changes as one character per position, "-" for None; non-finite min_depths keyed by name);
  cdr         `cdr_start_consensuses` / `cdr_end_consensuses` -> Regions for every (decay, mask_ends) of
              table_cases.CDR_OPTIONS;
  base / freq / tie   `consensus(w)` of every position's weights.
and, under "files", `bam_to_consensus` of two alignment fixtures under the min_depths whose ceiling is no int64
(FASTA, changes, reports with the input path replaced by "{path}").

The output is deterministic (gzip mtime 0, sorted keys): a second run writes the same bytes.
"""
from __future__ import annotations

import gzip
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import refload  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "table_runs.json.gz")
FILES = ("inputs/cut_bwa_1_1.bam", "inputs/cut_mm2_multi.bam")
FILE_MIN_DEPTHS = ("inf", "-inf", "nan", "1e19", "2.5")
_ORDER = "ATGCN"  # dict order of the reference's weight dicts (kindel.py:29)
_COL = {"A": 0, "C": 1, "G": 2, "T": 3, "N": 4}


def reference_inputs(case):
    c = case["counts"].tolist()
    L = case["L"]

    def dicts(c0):
        return [{k: c[c0 + _COL[k]][p] for k in _ORDER} for p in range(L)]

    def acgt(c0):
        return [sum(c[c0 + k][p] for k in range(4)) for p in range(L)]

    insertions = [dict(case["insertions"].get(s, [])) for s in range(L + 1)]
    return {"weights": dicts(0), "deletions": c[5][:L + 1], "insertions": insertions,
            "clip_start_weights": dicts(9), "clip_end_weights": dicts(14),
            "clip_start_depth": acgt(9), "clip_end_depth": acgt(14)}


def _changes(ch):
    return "".join("-" if x is None else x for x in ch)


def table_run(k, case):
    import table_cases as T

    r = reference_inputs(case)
    out = {"L": case["L"], "consensus": {}, "cdr": {}}
    for name, md in T.MIN_DEPTHS:
        seq, ch = k.consensus_sequence(r["weights"], r["insertions"], r["deletions"], None, False, md, False)
        out["consensus"][name] = [seq, _changes(ch)]
    for decay, mask in T.CDR_OPTIONS:
        f = k.cdr_start_consensuses(r["weights"], r["deletions"], r["clip_start_weights"], r["clip_start_depth"],
                                    decay, mask)
        e = k.cdr_end_consensuses(r["weights"], r["deletions"], r["clip_end_weights"], r["clip_end_depth"],
                                  decay, mask)
        out["cdr"][T.cdr_key(decay, mask)] = {"start": [list(x) for x in f], "end": [list(x) for x in e]}
    cons = [k.consensus(w) for w in r["weights"]]
    out["base"] = "".join(x[0] for x in cons)
    out["freq"] = [x[1] for x in cons]
    out["tie"] = "".join("1" if x[3] else "0" for x in cons)
    return out


def file_run(k, rel):
    import table_cases as T

    path = os.path.join(ROOT, "tests", "golden", rel)
    mds = dict(T.MIN_DEPTHS)
    out = {}
    for name in FILE_MIN_DEPTHS:
        res = k.bam_to_consensus(path, False, mds[name])
        out[name] = {"fasta": [[s.name, s.sequence] for s in res.consensuses],
                     "changes": {c: _changes(ch) for c, ch in res.refs_changes.items()},
                     "reports": {c: rep.replace(path, "{path}") for c, rep in res.refs_reports.items()}}
    return out


def main():
    import table_cases as T

    if not refload.available():
        raise SystemExit("no reference tree found; see oracle/refload.py")
    k = refload.load_reference()
    data = {"reference": "bede/kindel v1.2.1 @ 14d727b", "cases": {}, "files": {}}
    for seed in range(T.N_CASES):
        data["cases"][str(seed)] = table_run(k, T.table_case(seed))
    for rel in FILES:
        data["files"][rel] = file_run(k, rel)
    with gzip.GzipFile(OUT, "wb", mtime=0) as fh:
        fh.write(json.dumps(data, sort_keys=True, separators=(",", ":")).encode())
    print(OUT, os.path.getsize(OUT), "bytes")


if __name__ == "__main__":
    main()
