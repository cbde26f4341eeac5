"""The production render kernel keeps its packed node step: compiled for sm_100a (no GPU needed), the staged
instantiation (local stack) still issues all the slab arithmetic of node_step as FFMA2, with no scalar FFMA left in it,
and still fits in the 72 registers its 896-thread launch allows.  The shared-memory-stack plan packs tc and the far
planes and keeps the near planes scalar."""
import os
import shutil
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))

pytestmark = pytest.mark.skipif(shutil.which("nvcc") is None or shutil.which("nvdisasm") is None, reason="needs nvcc and nvdisasm")


@pytest.fixture(scope="module")
def census():
    import sass_census

    return sass_census.census(ROOT)


def test_production_node_step_is_packed(census):
    c = census["render_kernel<0,1,0,0,0,0>"]
    assert c["regs"] == 72
    assert c["step_FFMA2"] > 0
    assert c["step_FFMA"] == 0


def test_every_staged_instantiation_is_packed(census):
    staged = [k for k in census if k.split("<")[1].split(",")[1] == "1"]
    assert len(staged) >= 10
    for name in staged:
        sstack = name.split("<")[1].split(",")[2] == "1"
        assert census[name]["FFMA2"] == (12 if sstack else 18), name
