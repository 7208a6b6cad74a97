"""TEST / BENCH INFRASTRUCTURE ONLY -- stages the UNMODIFIED reference package inside the tree.

The reference (bede/kindel v1.2.1) is a pure-Python flit package whose run-time dependencies (simplesam,
dnaio, argh) need not be installed, so this recipe puts what a `pip install --target` would have put there
for a pure-Python package -- the package directory `kindel/` with its three modules, byte for byte -- and
nothing else under `oracle/_ref/`.  `oracle/_ref/` is git-ignored (never part of the repository's history);
it lets `bench.py --impl reference` / `cpu_baseline` time the reference's own `parse_records` +
`consensus_sequence` (reference kindel/kindel.py:21-128, 384-430) through `oracle/refload.py`'s import stubs
on a machine that has no reference checkout.

    python -m oracle.stage_reference          (also called by __graft_entry__.build(); a no-op without a source)
"""
from __future__ import annotations

import hashlib
import os
import shutil
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.environ.get("KINDEL_REFERENCE_SRC", "/root/reference")
DST = os.path.join(ROOT, "oracle", "_ref")
FILES = ("__init__.py", "kindel.py", "cli.py")


def stage(verbose: bool = False) -> str | None:
    """Copy <SRC>/kindel/*.py to oracle/_ref/kindel/.  Returns the staged root, or None if SRC is absent."""
    src_pkg = os.path.join(SRC, "kindel")
    if not os.path.isfile(os.path.join(src_pkg, "kindel.py")):
        return DST if os.path.isfile(os.path.join(DST, "kindel", "kindel.py")) else None
    dst_pkg = os.path.join(DST, "kindel")
    os.makedirs(dst_pkg, exist_ok=True)
    lines = []
    for f in FILES:
        s, d = os.path.join(src_pkg, f), os.path.join(dst_pkg, f)
        if not os.path.isfile(s):
            continue
        shutil.copyfile(s, d)
        with open(d, "rb") as fh:
            lines.append("%s  kindel/%s" % (hashlib.sha256(fh.read()).hexdigest(), f))
    with open(os.path.join(DST, "STAGED_FROM.txt"), "w") as fh:
        fh.write("staged from %s by oracle/stage_reference.py (unmodified)\n" % SRC)
        fh.write("\n".join(lines) + "\n")
    if verbose:
        print("\n".join(lines), file=sys.stderr)
    return DST


if __name__ == "__main__":
    print(stage(verbose=True))
