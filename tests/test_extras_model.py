"""CPU tests of the combined reference model (tests/extras_model.py): its best / web / runner_up are
runner_up_model.match_wta_ru's, its best / web / web_sub are subpixel_model.match_wta_sub's, its best / web at m = 0 are
the oracle's own winner-take-all, over both variants, both oracle paths, ranges that start past the frame's width and
ranges of more than 64 shifts; and the invariants that tie the outputs together hold."""
import numpy as np
import pytest

import stereomatching_b200 as smb
from extras_model import match_wta_all, reference_all
from runner_up_model import match_wta_ru
from subpixel_model import match_wta_sub
from util import vname

W, H, SW = 24, 12, 5


def maps(D, seed):
    rng = np.random.default_rng(seed)
    le = (rng.random((H, W)) < 0.4).astype(np.uint8)
    yield "random", le, np.roll(le, 3 + seed % 5, axis=1) ^ (rng.random((H, W)) < 0.05).astype(np.uint8)
    yield "noisy", le, (rng.random((H, W)) < 0.5).astype(np.uint8)
    yield "saturated", np.zeros((H, W), np.uint8), np.zeros((H, W), np.uint8)
    yield "no_match", np.ones((H, W), np.uint8), np.zeros((H, W), np.uint8)
    p = np.tile((rng.random((H, 8)) < 0.5).astype(np.uint8), (1, W // 8))
    yield "periodic8", p, p.copy()


@pytest.mark.parametrize("direct", [False, True], ids=["separable", "literal"])
@pytest.mark.parametrize("variant", [smb.WRAP, smb.GHOST], ids=vname)
@pytest.mark.parametrize("m", [0, 4, 37, W, 2 * W + 3])
@pytest.mark.parametrize("D", [1, 2, 17, 65, 130])
def test_model(orc, variant, direct, m, D):
    for name, le, re in maps(D, 7 * D + m):
        what = "%s D %d m %d" % (name, D, m)
        best, web, ru, ws = match_wta_all(orc, le, re, D, SW, variant, m=m, direct=direct)
        assert all(a.dtype == np.int32 and a.shape == (H, W) for a in (best, web, ru, ws)), what
        bo, wo, ro = match_wta_ru(orc, le, re, D, SW, variant, direct=direct, m=m)
        assert np.array_equal(best, bo) and np.array_equal(web, wo) and np.array_equal(ru, ro), what
        bs, wsw, so = match_wta_sub(orc, le, re, D, SW, variant, direct=direct, m=m)
        assert np.array_equal(best, bs) and np.array_equal(web, wsw) and np.array_equal(ws, so), what
        if m == 0:
            bw, ww = orc.match_wta(le, re, D, SW, variant, direct=direct)
            assert np.array_equal(best, bw) and np.array_equal(web, ww), what
        # the invariants
        assert (ru <= best).all(), what
        assert np.array_equal((ws + 8) >> 4, web), what
        assert ((web >= m + 1) & (web <= m + D)).all(), what
        ends = (web == m + 1) | (web == m + D)
        assert np.array_equal(ws[ends], 16 * web[ends]), what
        if D == 1:
            assert not ru.any() and np.array_equal(ws, 16 * web), what
        if name == "periodic8" and variant == smb.WRAP and D > 8 and m % 8 == 0:
            assert (ru == best).mean() > 0.5, what  # shifts 8 apart tie: the runner-up is best again


@pytest.mark.parametrize("variant", [smb.WRAP, smb.GHOST], ids=vname)
def test_reference_expands_equal_rows(orc, variant):
    """reference_all on maps whose rows are all equal (evaluated on 2*half+1 rows) is match_wta_all on the frame."""
    rng = np.random.default_rng(5 + variant)
    D, m, sw, Hb = 70, 9, 5, 30
    row = (rng.random(W) < 0.5).astype(np.uint8)
    le = np.tile(row, (Hb, 1))
    re = np.tile(np.roll(row, m + 20), (Hb, 1))
    want = match_wta_all(orc, le, re, D, sw, variant, m=m)
    got = reference_all(orc, "rows", le, re, D, sw, variant, m)
    for g, w in zip(got, want):
        assert np.array_equal(g, w)
