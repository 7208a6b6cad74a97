"""The offline kernel tools (tools/) keep working: opcode census of the built library, per-source-line ncu budget.
They need the CUDA toolkit's cuobjdump / nvdisasm / ncu but no GPU."""
import os
import shutil
import subprocess
import sys

import pytest

from helpers import ROOT

pytestmark = pytest.mark.skipif(shutil.which("cuobjdump") is None or shutil.which("nvdisasm") is None,
                                reason="needs the CUDA toolkit binaries")


def _run(*args):
    return subprocess.run([sys.executable, *args], cwd=ROOT, capture_output=True, text=True, timeout=600)


@pytest.mark.skipif(shutil.which("ncu") is None, reason="needs ncu")
def test_ncu_lines_on_a_saved_report():
    """KDL_NCU_REPORT: a report of the tile kernel captured with source counters, e.g.
    ncu --section SourceCounters --section WarpStateStats --import-source on -k regex:pileup_tile -c 1 -o k1_tile \
        python bench.py --workload tiny --steps 1 --no-cpu
    Such a report is 3.3 MB (0.4 MB xz-compressed), too large to keep in the repository as a test vector."""
    rep = os.environ.get("KDL_NCU_REPORT")
    if not rep:
        pytest.skip("set KDL_NCU_REPORT to a saved ncu report of the tile kernel")
    res = _run("tools/ncu_lines.py", rep, "10")
    assert res.returncode == 0, res.stderr
    assert "executed warp instructions" in res.stdout and "pileup_tile.cu" in res.stdout


def test_opcode_census_proves_the_design_claims():
    res = _run("tools/opcode_census.py")
    assert res.returncode == 0, res.stderr
    tile = [ln for ln in res.stdout.splitlines() if "pileup_tile_kernel" in ln]
    assert len(tile) == 6 and "sm_100a" in res.stdout
    for ln in tile:  # total, UBLKCP, SYNCS, LDGSTS, USETMAXREG ... UTCMMA, HMMA
        f = ln.split()
        nums = [int(x) for x in f[-18:]]
        assert nums[1] >= 1 and nums[2] >= 10 and nums[3] >= 10 and nums[4] == 2 and nums[-1] == 0 and nums[-2] == 0


def test_results_table_matches_the_readme():
    """README.md's results block is the output of tools/results_table.py over profiles/: it cannot drift."""
    res = _run("tools/results_table.py")
    assert res.returncode == 0, res.stderr
    lines = [ln for ln in res.stdout.splitlines() if ln.startswith("|")]
    assert len(lines) >= 8 and "cfg4_5Mb_200x" in res.stdout
    readme = open(os.path.join(ROOT, "README.md")).read()
    a = readme.index("<!-- results:begin")
    b = readme.index("<!-- results:end -->")
    block = readme[a:b].split("\n", 1)[1]
    assert block.strip() == res.stdout.strip()
