"""Static ALU-pipe budget of the kernel with both extras at config 2 (tools/sass_budget.py --family
k_bitslice_ru_sub), read from the SASS of the built library.  Pass A is the 16-bit kernel's walk unchanged.  Pass B
holds both families' epilogues on the same registers: at most the sum of their limits, 510 + 112 + 32 + 224 + 64 =
942 ALU-pipe instructions; the build reaches 941.  No GPU needed."""
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
    return {f: sass_budget.budget(LIB, (4, 2, 16, 0, 0, 0), f) for f in ("k_bitslice16", "k_bitslice_ru_sub")}


def test_pass_a_walk(budgets):
    """The walk's ALU-pipe work is the sibling's, opcode for opcode (ptxas schedules one IMAD fewer into it)."""
    a, a16 = budgets["k_bitslice_ru_sub"]["pass_a"], budgets["k_bitslice16"]["pass_a"]
    assert a["alu"] == a16["alu"] and a["alu_ops"] == a16["alu_ops"]
    assert a["lsu"] == a16["lsu"] and a["fma"] <= a16["fma"]


def test_pass_b_block(budgets):
    b, b16 = budgets["k_bitslice_ru_sub"]["pass_b"], budgets["k_bitslice16"]["pass_b"]
    assert b["alu_ops"].get("FLO", 0) <= b16["alu_ops"].get("FLO", 0)
    assert b["alu_ops"].get("LEA", 0) == 0  # power-of-two multiplies stay multiply-adds
    assert b["alu"] <= 941
    assert b["alu"] <= 510 + 112 + 32 + 224 + 64
