"""SASS budget of the fused GMW forward's converter step loops (compiled for sm_100a here; no GPU needed).

Every mlp_fused_kernel<UPO> instantiation must stay within 128 registers (512 threads, one CTA per SM) without spills or
local memory in its step loops.  The common path of a steady-state step (profiles/sass_fused.py) is held to what it is
now, so that an edit which puts work back on the converters' path shows here before it shows on the GPU.
"""
import importlib.util
import os
import shutil

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NVCC = os.environ.get("NVCC") or ("/usr/local/cuda/bin/nvcc" if os.path.exists("/usr/local/cuda/bin/nvcc") else shutil.which("nvcc"))

pytestmark = pytest.mark.skipif(not NVCC, reason="nvcc not found")

# common-path budget of a steady-state step in the full-slice loops (warp-instructions per 16-edge unit), by kind and by
# steps per loop iteration (the loop is unrolled by two except at UPO = 4, which would spill)
BUDGET = {("kind0", 2): 175, ("kind0", 1): 200, ("kind2", 2): 150, ("kind2", 1): 150}


@pytest.fixture(scope="module")
def report():
    spec = importlib.util.spec_from_file_location("sass_fused", os.path.join(ROOT, "profiles", "sass_fused.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.analyse()


def test_every_slice_geometry_is_instantiated_without_spills(report):
    assert sorted(report) == [3, 4, 5, 6, 7]
    for upo, r in report.items():
        assert r["registers"] <= 128, upo
        assert r["spill_stores"] == 0 and r["spill_loads"] == 0, upo


def test_step_loops_fit_their_budget(report):
    for upo, r in report.items():
        loops = r["step_loops"]
        # one full-slice and one tail loop per kind: a budget cannot be skipped because a variant went missing
        assert sorted((lp["kind"], lp["variant"]) for lp in loops) == [
            (k, v) for k in ("first", "kind0", "kind2") for v in ("full", "tail")], upo
        for lp in loops:
            assert lp["local_memory"] == 0, (upo, lp["kind"], lp["variant"])
            if lp["kind"] != "first" and lp["variant"] == "full":
                assert lp["common_path"] <= BUDGET[(lp["kind"], lp["steps"])], (upo, lp["kind"], lp["common_path"])
