"""Static ALU-pipe budget of the hot kernel's steady blocks at config 2 (tools/sass_budget.py), read from the SASS
of the built library.  The kernel is bound by the ALU pipe; this guards against an edit that quietly gives
instructions back (ptxas re-associating the bit-plane logic, a select falling back from the FMA pipe to a SEL).
No GPU needed."""
import os
import shutil
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "stereomatching_b200", "libstereo_b200.so")

pytestmark = pytest.mark.skipif(not os.path.exists(LIB) or shutil.which("cuobjdump") is None,
                                reason="needs the built library and cuobjdump")


@pytest.fixture(scope="module")
def budget():
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    try:
        import sass_budget
    finally:
        sys.path.pop(0)
    return sass_budget.budget(LIB, (4, 2, 16, 0, 0, 0))


def test_pass_a_walk(budget):
    # 16 counter steps x 7 LOP3 + the fill's carry-save tree, and no SEL: the complement is a predicated IMAD
    a = budget["pass_a"]
    assert a["alu_ops"].get("SEL", 0) <= 1
    assert a["alu_ops"]["LOP3"] <= 130
    assert a["alu"] <= 158


def test_pass_b_block(budget):
    # 8 rows x 2 words x 21 LOP3 of the add/sub ripple + 112 of the winner-take-all + one per row
    b = budget["pass_b"]
    assert b["alu_ops"]["LOP3"] <= 8 * 2 * 21 + 112 + 8
    assert b["alu_ops"].get("SEL", 0) <= 8
    assert b["alu"] <= 510


def test_per_pixel(budget):
    assert budget["pixels_per_warp_block"] == 256
    assert budget["alu_per_pixel"]["steady"] <= 83.0
