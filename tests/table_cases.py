"""Seeded adversarial count tables for the kernels that turn a finished table into the answer (test infrastructure):
K2 / K2p / K2x (vote), K2d (derived columns), K4 (--realign flags) and K5 (consensus text).

Tables that come from pileups of reads almost never sit on the decision boundaries of those kernels.  These do:

  small counts       every column in {0..3} with about 40 % zeros: base ties, exact halves, N-only and empty slots;
  planted boundaries at slots p = 3 (mod 4) (the look-ahead depth comes from the next lane), p = 127 (mod 128) (lane 31
                     reloads it), p = 1023 (mod 1024) (CTA edge) and at the last position L - 1 of the contig:
                       2 ins == min(d, dn) or min(d, dn) + 1 with dn < d (the look-ahead decides),
                       2 del == depth or depth + 1, depth == ceil(md) - 1 or ceil(md) for the stored min_depths,
                       N-only and all-zero positions;
  K4 thresholds      for every decay of DECAYS, tot = weights + deletions and clip depth cd with tot * decay equal to cd
                     after rounding in double, or one ulp either side; 2 cd == tot + 1 and tot + 2; some tot near 2**24;
  insertion dicts    1-3 distinct strings of length 1-300 per insertion slot, counts summing to column 6, in a stated
                     first-seen order, with ties among them.

A case is one contig of length L: `counts` int32 [19, L + 1] in the engine's column layout (include/kindel_b200.h:
0-4 weights A,C,G,T,N, 5 deletions, 6 insertion total, 7 / 8 clip starts / ends, 9-13 / 14-18 clip start / end weights
A,C,G,T,N) and `insertions` {slot: [(string, count), ...]}.  Slot L is zero in columns 0-4, as a pileup leaves it;
columns 5, 6 and 7-18 may be non-zero there.  `pack` lays several cases out in one table.

`large_table` is the large tier: counts up to 2**24 at random places of a big table.  The kernels' derived int32 sums
(five weights + deletions, four clip weights) assume every count is at most 2**28; nothing here goes above 2**24.
"""
from __future__ import annotations

import math
import random

import numpy as np

N_CASES = 44
LONG_L = {40: 1023, 41: 1024, 42: 1025, 43: 2049}  # the rest have L <= 300
MIN_DEPTHS = (("0", 0), ("1", 1), ("2", 2), ("2.5", 2.5), ("7", 7), ("inf", math.inf), ("-inf", -math.inf),
              ("nan", math.nan), ("1e19", 1e19))
CDR_OPTIONS = ((0.1, 50), (0.1, 0), (0.3, 3), (1 / 3, 1), (0.0, 5), (0.7, 2))  # (clip_decay_threshold, mask_ends)
DECAYS = (0.1, 0.3, 1 / 3, 0.7, 0.0, 0.5, 1.0)
_DENOM = {0.1: 10, 0.3: 10, 1 / 3: 3, 0.7: 10, 0.0: 1, 0.5: 2, 1.0: 1}
_ALPHABET = "ACGTN"


def cdr_key(decay, mask_ends):
    return "%r/%d" % (decay, mask_ends)


def _split(rng, total, parts):
    """`total` as `parts` non-negative ints."""
    cuts = sorted(rng.randint(0, total) for _ in range(parts - 1))
    return [b - a for a, b in zip([0] + cuts, cuts + [total])]


def _set_depth(rng, counts, s, depth, n_extra=None):
    """ACGT weights of slot s summing to `depth` (N weight random unless given)."""
    counts[0:4, s] = _split(rng, depth, 4)
    counts[4, s] = rng.choice([0, 0, 1, 2]) if n_extra is None else n_extra


def plant_ins_boundary(rng, counts, p, at_limit, free_next=True, dn=None):
    """Slot p: an insertion decision that only the look-ahead depth dn of slot p + 1 (dn < d) decides.  at_limit:
    2 ins == dn (no call; dn - 1 if dn is odd), else 2 ins == dn + 1 (a call; dn + 2 if dn is even).  free_next:
    slot p + 1 gets a fresh depth dn (random of the right parity unless given), else its depth stays (the extra slot
    of a contig: 0)."""
    if free_next:
        if dn is None:
            dn = 2 * rng.randint(0, 3) + (0 if at_limit else 1)
        _set_depth(rng, counts, p + 1, dn)
    else:
        dn = int(counts[0:4, p + 1].sum())
    d = dn + rng.randint(1, 6)
    _set_depth(rng, counts, p, d)
    counts[5, p] = rng.randint(0, d // 2)
    counts[6, p] = dn // 2 if at_limit else dn // 2 + 1


def _plant(rng, counts, p, kind, L):
    if kind == "ins":
        plant_ins_boundary(rng, counts, p, rng.random() < 0.5, free_next=p + 1 < L)
    elif kind == "del":
        d = rng.randint(0, 9)
        _set_depth(rng, counts, p, d)
        counts[5, p] = (d + 1) // 2  # 2 del == d (d even: no D) or d + 1 (d odd: D)
    elif kind == "depth":
        _set_depth(rng, counts, p, rng.choice([0, 1, 1, 2, 2, 3, 3, 6, 7]))
        counts[5, p] = 0
    elif kind == "nonly":
        counts[0:4, p] = 0
        counts[4, p] = rng.randint(1, 3)
        counts[5, p] = rng.randint(0, 1)
    else:  # "zero"
        counts[0:7, p] = 0


def _plant_k4(rng, counts, p):
    """Slot p: tot = five weights + deletions and a clip depth cd on the edge of one K4 predicate."""
    decay = rng.choice(DECAYS)
    big = rng.random() < 0.3
    if rng.random() < 0.35:  # dominance: 2 cd == tot + 1 (not dominant) or tot + 2 (dominant)
        tot = rng.randint(1, 2 ** 24) if big else rng.randint(1, 40)
        cd = (tot + 1 + rng.randint(0, 1) + 1) // 2
    else:  # decay: tot * decay == cd after rounding in double, or an ulp either side
        if big:
            tot = rng.randint(2 ** 20, 2 ** 24)
        else:
            tot = _DENOM[decay] * rng.randint(0, 12)
        cd = max(0, int(round(tot * decay)) + rng.choice([-1, 0, 0, 1]))
        cd = min(cd, 4 * 2 ** 24)
    dele = rng.randint(0, tot) if rng.random() < 0.5 else 0
    w = _split(rng, tot - dele, 5)
    while max(w) > 2 ** 24:  # keep every count <= 2**24: move the excess into the deletions
        k = w.index(max(w))
        dele += w[k] - 2 ** 24
        w[k] = 2 ** 24
    if dele > 2 ** 24:
        return
    counts[0:5, p] = w
    counts[5, p] = dele
    c0 = rng.choice([9, 14])
    cw = _split(rng, cd, 4)
    if max(cw) > 2 ** 24:
        return
    counts[c0:c0 + 4, p] = cw
    counts[c0 + 4, p] = rng.choice([0, 0, 1, 3])


def _insertion_dict(rng, total):
    n = rng.randint(1, min(3, total))
    if n > 1 and rng.random() < 0.4:  # ties between the strings
        share = total // n
        parts = [share] * n
        parts[-1] += total - share * n
    else:
        parts = [x + 1 for x in _split(rng, total - n, n)]
    strings = []
    while len(strings) < n:
        ln = rng.randint(1, 300) if rng.random() < 0.05 else rng.randint(1, 4)
        s = "".join(rng.choice(_ALPHABET) for _ in range(ln))
        if s not in strings:
            strings.append(s)
    return list(zip(strings, parts))


def table_case(seed):
    """-> dict(L, counts int32 [19, L + 1], insertions {slot: [(string, count), ...]})."""
    rng = random.Random(70_000 + seed)
    if seed in LONG_L:
        L = LONG_L[seed]
    elif seed % 5 == 0:
        L = rng.choice([1, 2, 3, 4, 5, 7, 8, 33])
    else:
        L = rng.randint(1, 300)
    n = L + 1
    counts = np.zeros((19, n), dtype=np.int64)
    for c in range(19):
        hi = L if c < 5 else n
        counts[c, :hi] = [0 if rng.random() < 0.4 else rng.randint(1, 3) for _ in range(hi)]
    kinds = ("ins", "ins", "del", "depth", "nonly", "zero")
    spots = {L - 1}
    spots.update(p for p in range(3, L, 4) if rng.random() < 0.3)
    spots.update(range(127, L, 128))
    spots.update(range(1023, L, 1024))
    for p in sorted(spots):
        _plant(rng, counts, p, rng.choice(kinds), L)
    for p in rng.sample(range(L), min(L, 1 + L // 12)):
        _plant_k4(rng, counts, p)
    counts = counts.astype(np.int32)
    insertions = {s: _insertion_dict(rng, int(counts[6, s])) for s in range(n) if counts[6, s] > 0}
    return {"L": L, "counts": counts, "insertions": insertions}


def pack(cases, rng, align=None):
    """Cases side by side in one table: (counts int32 [19, n_slots], contig_slot int64, contig_len int32, insertions
    {slot: dict}).  align=None: arbitrary starts (random gaps of 0-5 slots); else every contig starts at a multiple of
    `align`.  n_slots is a multiple of 4 with at least one padding slot."""
    starts, s = [], 0
    for c in cases:
        s = -(-s // align) * align if align else s + rng.randint(0, 5)
        starts.append(s)
        s += c["L"] + 1
    n_slots = (s + 4) // 4 * 4
    counts = np.zeros((19, n_slots), dtype=np.int32)
    ins = {}
    for st, c in zip(starts, cases):
        counts[:, st:st + c["L"] + 1] = c["counts"]
        for k, v in c["insertions"].items():
            ins[st + k] = dict(v)
    return counts, np.array(starts, dtype=np.int64), np.array([c["L"] for c in cases], dtype=np.int32), ins


def large_table(seed, n_slots, n_hot=20_000):
    """The large tier: a table of n_slots (multiple of 4) with small counts everywhere and counts up to 2**24 at
    n_hot random slots (weights, deletions, insertions, clip weights)."""
    rng = np.random.default_rng(seed)
    counts = np.empty((19, n_slots), dtype=np.int32)
    for c in range(19):
        col = rng.integers(1, 4, size=n_slots, dtype=np.int32)
        col[rng.random(n_slots, dtype=np.float32) < 0.4] = 0
        counts[c] = col
    counts[0:5, -1] = 0
    hot = rng.choice(n_slots - 1, size=n_hot, replace=False)
    for c in (0, 1, 2, 3, 4, 5, 6, 9, 10, 11, 12, 14, 15, 16, 17):
        pick = hot[rng.random(n_hot) < 0.5]
        counts[c, pick] = rng.integers(0, 2 ** 24 + 1, size=pick.shape[0], dtype=np.int32)
    return counts
