"""Static ALU-pipe budget of the runner-up kernel's steady blocks at config 2 (tools/sass_budget.py --family
k_bitslice_ru), read from the SASS of the built library.  Pass A is the int32 kernel's walk unchanged; pass B adds
the second bit-serial max of the winner-take-all (one LOP3 per plane and word: 8 rows x 2 words x 7 planes = 112),
the lanes it runs over (one LOP3 per word: 16) and the runner-up store, and at most 510 + 112 + 32 = 654 ALU-pipe
instructions in all.  No GPU needed."""
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
    return {f: sass_budget.budget(LIB, (4, 2, 16, 0, 0, 0), f) for f in ("k_bitslice16", "k_bitslice_ru")}


def test_pass_a_walk(budgets):
    a = budgets["k_bitslice_ru"]["pass_a"]
    assert a["alu_ops"].get("SEL", 0) <= 1
    assert a["alu_ops"]["LOP3"] <= 130
    assert a["alu"] <= 158
    assert a == budgets["k_bitslice16"]["pass_a"]


def test_pass_b_block(budgets):
    b, b16 = budgets["k_bitslice_ru"]["pass_b"], budgets["k_bitslice16"]["pass_b"]
    # the second chain and the dropped tied lane: 112 + 16 LOP3 (the negation is on the FMA pipe), no shift and no
    # FLO of their own
    assert b["alu_ops"]["LOP3"] <= b16["alu_ops"]["LOP3"] + 112 + 16
    assert b["alu_ops"].get("SHF", 0) <= b16["alu_ops"].get("SHF", 0)
    assert b["alu_ops"]["FLO"] == b16["alu_ops"]["FLO"]
    assert b["alu"] <= 510 + 112 + 32


def test_pass_b_ring_slots_stay_off_the_alu_pipe(budgets):
    # the centre-match rows of a steady block are consecutive ring rows: no per-row compare-and-select on the ALU pipe
    b, b16 = budgets["k_bitslice_ru"]["pass_b"], budgets["k_bitslice16"]["pass_b"]
    assert b["alu_ops"].get("ISETP", 0) <= b16["alu_ops"].get("ISETP", 0)
    assert b["alu_ops"].get("SEL", 0) <= 2 * b16["alu_ops"].get("SEL", 0)
