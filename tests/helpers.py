"""Shared helpers for the parity tests (test infrastructure)."""
from __future__ import annotations

import gzip
import hashlib
import json
import os
import sys
from collections import OrderedDict

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

NIBBLES = "=ACMGRSVTWYHKDBN"
BASES = "ACGTN"
NCOL = 19


def reference_alignment_to_table(aln):
    """Reference `alignment` namedtuple (kindel/kindel.py:97-128) -> (counts[19, L+1], ins dicts)."""
    L = len(aln.weights)
    t = np.zeros((NCOL, L + 1), dtype=np.int64)
    for k, b in enumerate(BASES):
        t[k, :L] = [w[b] for w in aln.weights]
        t[9 + k, :L] = [w[b] for w in aln.clip_start_weights]
        t[14 + k, :L] = [w[b] for w in aln.clip_end_weights]
    t[5] = aln.deletions
    t[6] = [sum(d.values()) for d in aln.insertions]
    t[7] = aln.clip_starts
    t[8] = aln.clip_ends
    ins = [OrderedDict(d) for d in aln.insertions]
    return t, ins


_reference_runs = None


def reference_runs():
    """What the unmodified reference returned on the seeded fuzz inputs and the FASTA files of its suite
    (tests/golden/reference_runs.json.gz, written by oracle/make_reference_golden.py)."""
    global _reference_runs
    if _reference_runs is None:
        with gzip.open(os.path.join(ROOT, "tests", "golden", "reference_runs.json.gz"), "rt") as fh:
            _reference_runs = json.load(fh)
    return _reference_runs


def table_sha256(table) -> str:
    """sha256 of a count table as int32 bytes (the layout of reference_alignment_to_table)."""
    return hashlib.sha256(np.ascontiguousarray(table, dtype=np.int32).tobytes()).hexdigest()


def frame_sha256(df) -> str:
    """sha256 of a DataFrame's column names, dtypes, index and values: equal digests <=> exactly equal frames."""
    h = hashlib.sha256()
    h.update(repr([(str(c), str(t)) for c, t in df.dtypes.items()]).encode())
    h.update(repr((str(df.index.dtype), df.index.tolist())).encode())
    for c in df.columns:
        v = df[c].to_numpy()
        h.update(repr(v.tolist()).encode() if v.dtype == object else np.ascontiguousarray(v).tobytes())
    return h.hexdigest()


def reference_lists(table, L):
    """int [19, L+1] table -> the reference's per-position lists (kindel/kindel.py:29-38, 91-96): weights,
    deletions, clip_start_weights, clip_end_weights, clip_start_depth, clip_end_depth."""
    t = np.asarray(table).tolist()

    def dicts(row0):
        return [{b: t[row0 + "ACGTN".index(b)][i] for b in "ATGCN"} for i in range(L)]

    csw, cew = dicts(9), dicts(14)
    return (dicts(0), t[5], csw, cew, [sum(w[b] for b in "ACGT") for w in csw], [sum(w[b] for b in "ACGT") for w in cew])


def event_string(batch, read, q_off, length):
    """Upper-case inserted string of one event, straight from the packed bases."""
    lseq = int(batch.seq_len[read])
    base = int(batch.seq_off[read])
    out = []
    for q in range(q_off, min(q_off + length, lseq)):
        w = int(batch.seq4[base + (q >> 3)])
        out.append(NIBBLES[(w >> (28 - 4 * (q & 7))) & 0xF])
    return "".join(out)


def events_to_dicts(batch, events):
    """Insertion event rows (slot, read, q_off, len) in iteration order -> {slot: OrderedDict}."""
    out = {}
    for slot, read, q_off, length in np.asarray(events).tolist():
        d = out.setdefault(slot, OrderedDict())
        s = event_string(batch, read, q_off, length)
        d[s] = d.get(s, 0) + 1
    return out


def contig_view(batch, table, c):
    """Slice of a [k, n_slots] table belonging to contig c: [k, L+1]."""
    s = int(batch.contig_slot[c])
    L = int(batch.contig_len[c])
    return table[..., s:s + L + 1]


def calls_to_changes(calls_slice):
    """calls bytes of one contig (length L) -> list of None/'D'/'N'/'I' like reference `changes`."""
    lut = [None, "D", "N", "I"]
    return [lut[(int(c) >> 4) & 3] for c in calls_slice]
