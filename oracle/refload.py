"""TEST INFRASTRUCTURE ONLY -- loads the UNMODIFIED reference (bede/kindel) for pinning the oracle.

This module exists only in service of the golden-data generators (`oracle/make_*golden.py`) and of
`bench.py`'s CPU legs: it imports `kindel/kindel.py` of a reference checkout (KINDEL_REFERENCE_ROOT)
exactly as it lies on disk (never copied into this repo) by stubbing the three third-party imports that
need not be installed (`simplesam`, `dnaio`, `argh`; reference `kindel/kindel.py:3,9,14`, `kindel/cli.py:2`) and
by feeding it records from a small stdlib (gzip + struct) BAM/SAM decoder that produces the four
attributes the pileup consumes (`.pos`, `.mapped`, `.seq`, `.cigars`; reference
`kindel/kindel.py:42-48`) plus `.rname` (`kindel/kindel.py:145`).

Where no reference checkout exists, the only copy is the staged install under `oracle/_ref/`
(git-ignored; `oracle/stage_reference.py`), used solely by `bench.py`'s CPU legs (`--impl reference`,
`cpu_baseline`) to time the reference's own functions; the tests and `smoke()` never import this module (they
compare with the reference's stored results under tests/golden/).  `available()` says whether a reference tree was found.

The decoder here is deliberately independent of the product decoder in `kindel_b200/bamio.py`
(record-at-a-time `struct.unpack`, no numpy), so the two cross-check each other.
"""
from __future__ import annotations

import importlib.util
import os
import sys
import types

_HERE = os.path.dirname(os.path.abspath(__file__))
# search order: explicit override, the reference tree of the build container, the staged install that
# stays with the tree (oracle/_ref/, produced by oracle/stage_reference.py; git-ignored)
_CANDIDATES = [os.environ.get("KINDEL_REFERENCE_ROOT"), "/root/reference",
               os.path.join(_HERE, "_ref")]


def _find_root():
    for c in _CANDIDATES:
        if c and os.path.isfile(os.path.join(c, "kindel", "kindel.py")):
            return c
    return "/root/reference"


REFERENCE_ROOT = _find_root()
_PKG = "_kindel_reference"  # private package name so it never shadows a user's `kindel`

from .samdecode import Record, read_alignment_file, read_bam, read_sam  # noqa: F401


def available() -> bool:
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "kindel", "kindel.py"))


class _Reader:
    """Stub for simplesam.Reader(fh): `.header` + iteration (kindel/kindel.py:137-145)."""

    def __init__(self, fh):
        self.header, self._records = read_alignment_file(fh.name)

    def __iter__(self):
        return iter(self._records)


class _Sequence:
    """Stub for dnaio.Sequence (kindel/kindel.py:434; consumed at kindel/cli.py:32-33)."""

    def __init__(self, name=None, sequence=None, qualities=None):
        self.name, self.sequence, self.qualities = name, sequence, qualities


_cached = None


def load_reference():
    """Return the reference module `kindel.kindel`, executed unmodified from REFERENCE_ROOT."""
    global _cached
    if _cached is not None:
        return _cached
    if not available():
        raise FileNotFoundError("reference tree not present at %s" % REFERENCE_ROOT)
    saved = {k: sys.modules.get(k) for k in ("simplesam", "dnaio", "argh")}
    simplesam = types.ModuleType("simplesam")
    simplesam.Reader = _Reader
    dnaio = types.ModuleType("dnaio")
    dnaio.Sequence = _Sequence
    argh = types.ModuleType("argh")
    sys.modules.update(simplesam=simplesam, dnaio=dnaio, argh=argh)
    try:
        pkg = types.ModuleType(_PKG)
        pkg.__path__ = []  # mark as package
        pkg.__version__ = "1.2.1"  # kindel/__init__.py:3
        cli = types.ModuleType(_PKG + ".cli")
        cli.main = lambda: None
        pkg.cli = cli
        sys.modules[_PKG] = pkg
        sys.modules[_PKG + ".cli"] = cli
        spec = importlib.util.spec_from_file_location(
            _PKG + ".kindel", os.path.join(REFERENCE_ROOT, "kindel", "kindel.py")
        )
        mod = importlib.util.module_from_spec(spec)
        sys.modules[_PKG + ".kindel"] = mod
        spec.loader.exec_module(mod)
        # silence the two tqdm bars (kindel/kindel.py:40,390): same iteration, no stderr noise
        class _Quiet:
            @staticmethod
            def tqdm(it, *a, **k):
                return it

        mod.tqdm = _Quiet
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    # the stubs must stay reachable from the module's globals (they are: bound at import time)
    _cached = mod
    return mod
