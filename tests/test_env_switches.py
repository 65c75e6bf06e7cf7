"""The library reads a short, documented list of environment variables (DESIGN.md §5a.5): test seams that select a
form giving the default's bits, and the switches bench.py sets.  A new "OFC_..." literal in the library's sources is a
new switch; it fails here until it is added to that list or removed."""
import os
import re

from tests.conftest import ROOT

PKG = os.path.join(ROOT, "opticalflowclustering_b200")

DOCUMENTED = {
    # test seams
    "OFC_TMEM_SHARE", "OFC_UPSAMPLE_X2", "OFC_POLY_STAGE", "OFC_PREFILTER_PYR",
    "OFC_KMEANS_TC", "OFC_KMEANS_FUSED", "OFC_KMEANS_MEDIUM", "OFC_CELLS_FAST",
    # benchmark switches
    "OFC_KMEANS_GRAPH", "OFC_KMEANS_PEER",
}


def _library_literals():
    found = {}
    for d, _, files in os.walk(PKG):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh")):
                path = os.path.join(d, f)
                with open(path, encoding="utf-8") as fh:
                    for name in re.findall(r"""["'](OFC_\w+)["']""", fh.read()):
                        found.setdefault(name, []).append(os.path.relpath(path, ROOT))
    return found


def test_library_reads_only_the_documented_environment_variables():
    found = _library_literals()
    assert set(found) == DOCUMENTED, {"undocumented": {n: found[n] for n in set(found) - DOCUMENTED},
                                      "no longer read": sorted(DOCUMENTED - set(found))}


def test_documented_list_is_in_design():
    with open(os.path.join(ROOT, "DESIGN.md"), encoding="utf-8") as fh:
        design = fh.read()
    assert [n for n in sorted(DOCUMENTED) if f"`{n}" not in design] == []
