"""CPU tests of the runner-up reference model (tests/runner_up_model.py): it is the second-largest value of the
stack of the oracle's score planes over the shifts (0 for one shift), and its best / web are the oracle's."""
import numpy as np
import pytest

from runner_up_model import match_wta_ru
from util import vname

import stereomatching_b200 as smb


def maps(W, H, D, seed):
    rng = np.random.default_rng(seed)
    le = (rng.random((H, W)) < 0.4).astype(np.uint8)
    yield "random", le, np.roll(le, 3, axis=1) ^ (rng.random((H, W)) < 0.05).astype(np.uint8)
    yield "saturated", np.zeros((H, W), np.uint8), np.zeros((H, W), np.uint8)
    yield "no_match", np.ones((H, W), np.uint8), np.zeros((H, W), np.uint8)
    p = np.tile((rng.random((H, 8)) < 0.5).astype(np.uint8), (1, W // 8))
    yield "periodic8", p, p.copy()


@pytest.mark.parametrize("direct", [False, True], ids=["separable", "literal"])
@pytest.mark.parametrize("variant", [smb.WRAP, smb.GHOST], ids=vname)
@pytest.mark.parametrize("D,sw,m", [(1, 5, 0), (2, 3, 0), (12, 5, 0), (20, 7, 0), (9, 5, 4)])
def test_second_order_statistic(orc, variant, direct, D, sw, m):
    W, H = 32, 20
    for name, le, re in maps(W, H, D, 100 * D + sw):
        best, web, ru = match_wta_ru(orc, le, re, D, sw, variant, direct=direct, m=m)
        scores = np.stack([orc.shift_planes(le, re, sw, m + i, variant, direct)[2] for i in range(D)])
        want = np.sort(scores, axis=0)[-2] if D >= 2 else np.zeros((H, W), np.int32)
        assert np.array_equal(ru, want), (name, D, sw)
        assert (ru <= best).all()
        # runner_up == best exactly where two shifts tie for best
        ties = (scores == best[None]).sum(axis=0) >= 2
        assert np.array_equal(ru == best, ties if D >= 2 else best == 0), name
        if m == 0:
            bo, wo = orc.match_wta(le, re, D, sw, variant, direct=direct)
            assert np.array_equal(best, bo) and np.array_equal(web, wo), name
        else:
            assert np.array_equal(best, scores.max(axis=0))
            assert np.array_equal(web, m + D - np.argmax(scores[::-1] == best[None], axis=0)), name
    if D == 1:
        assert not ru.any()


def test_saturated_maps_tie_everywhere(orc):
    W, H, D, sw = 24, 16, 6, 5
    z = np.zeros((H, W), np.uint8)
    best, web, ru = match_wta_ru(orc, z, z, D, sw, smb.WRAP, direct=True)
    assert (best == sw * sw).all() and (ru == sw * sw).all() and (web == D).all()
