"""Static ALU-pipe budget of the sub-pixel kernel's steady blocks at config 2 (tools/sass_budget.py --family
k_bitslice_sub), read from the SASS of the built library.  Pass A is the 16-bit kernel's walk unchanged; pass B adds
the gather of the winner's two neighbour scores (one LOP3 per plane, word and neighbour: 8 rows x 2 x 2 x 7 = 224),
the two shifts that place the winner's bit in each word (16), and the four compares of the fraction's search (32); the
rest of it runs on the FMA pipe.  At most 510 + 2 * 112 + 64 = 798 ALU-pipe instructions in all; the build reaches
793.  No GPU needed."""
import os
import shutil
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "stereomatching_b200", "libstereo_b200.so")

pytestmark = pytest.mark.skipif(not os.path.exists(LIB) or shutil.which("cuobjdump") is None,
                                reason="needs the built library and cuobjdump")


@pytest.fixture(scope="module")
def budgets():
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    try:
        import sass_budget
    finally:
        sys.path.pop(0)
    return {f: sass_budget.budget(LIB, (4, 2, 16, 0, 0, 0), f) for f in ("k_bitslice16", "k_bitslice_sub")}


def test_pass_a_walk(budgets):
    assert budgets["k_bitslice_sub"]["pass_a"] == budgets["k_bitslice16"]["pass_a"]


def test_pass_b_block(budgets):
    b, b16 = budgets["k_bitslice_sub"]["pass_b"], budgets["k_bitslice16"]["pass_b"]
    assert b["alu_ops"]["LOP3"] <= b16["alu_ops"]["LOP3"] + 224
    assert b["alu_ops"].get("FLO", 0) <= b16["alu_ops"].get("FLO", 0)
    assert b["alu_ops"].get("SHF", 0) <= b16["alu_ops"].get("SHF", 0) + 16
    assert b["alu_ops"].get("LEA", 0) == 0  # power-of-two multiplies stay multiply-adds
    assert b["alu"] <= 793
    assert b["alu"] <= 510 + 2 * 112 + 64
