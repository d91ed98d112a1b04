"""CPU tests of the sub-pixel reference model (tests/subpixel_model.py): its best / web are the oracle's, its
web_sub is the parabola vertex of the contract (checked against a float64 restatement), and the invariants hold."""
import numpy as np
import pytest

from subpixel_model import match_wta_sub, sub_frac
from util import vname

import stereomatching_b200 as smb


def maps(W, H, D, seed):
    rng = np.random.default_rng(seed)
    le = (rng.random((H, W)) < 0.4).astype(np.uint8)
    yield "random", le, np.roll(le, 3, axis=1) ^ (rng.random((H, W)) < 0.05).astype(np.uint8)
    yield "noisy", le, (rng.random((H, W)) < 0.4).astype(np.uint8)
    yield "saturated", np.zeros((H, W), np.uint8), np.zeros((H, W), np.uint8)
    yield "no_match", np.ones((H, W), np.uint8), np.zeros((H, W), np.uint8)
    p = np.tile((rng.random((H, 8)) < 0.5).astype(np.uint8), (1, W // 8))
    yield "periodic8", p, p.copy()


def float_web_sub(scores, m):
    """The contract restated in float64: the vertex (s+ - s-) / (2 den) in sixteenths, rounded half up, clamped to 7,
    0 at the range ends."""
    D = scores.shape[0]
    best = scores.max(axis=0)
    w = D - 1 - np.argmax(scores[::-1] == best[None], axis=0)
    out = 16.0 * (m + w + 1)
    for idx in np.ndindex(best.shape):
        k = w[idx]
        if 0 < k < D - 1:
            sm, s0, sp = (float(scores[(j,) + idx]) for j in (k - 1, k, k + 1))
            frac = min(7.0, np.floor(16.0 * (sp - sm) / (2.0 * (2.0 * s0 - sm - sp)) + 0.5))
            out[idx] += frac
    return out


@pytest.mark.parametrize("direct", [False, True], ids=["separable", "literal"])
@pytest.mark.parametrize("variant", [smb.WRAP, smb.GHOST], ids=vname)
@pytest.mark.parametrize("D,sw,m", [(1, 5, 0), (2, 3, 0), (3, 3, 0), (12, 5, 0), (20, 7, 0), (9, 5, 4)])
def test_model(orc, variant, direct, D, sw, m):
    W, H = 32, 20
    for name, le, re in maps(W, H, D, 100 * D + sw):
        best, web, ws = match_wta_sub(orc, le, re, D, sw, variant, direct=direct, m=m)
        scores = np.stack([orc.shift_planes(le, re, sw, m + i, variant, direct)[2] for i in range(D)])
        if m == 0:
            bo, wo = orc.match_wta(le, re, D, sw, variant, direct=direct)
            assert np.array_equal(best, bo) and np.array_equal(web, wo), name
        else:
            assert np.array_equal(best, scores.max(axis=0))
            assert np.array_equal(web, m + D - np.argmax(scores[::-1] == best[None], axis=0)), name
        assert np.array_equal(ws, float_web_sub(scores, m)), name
        # the invariants
        assert np.array_equal((ws + 8) >> 4, web), name
        assert (ws >= 16 * (m + 1) - 8).all() and (ws > 0).all() and (ws < 1 << 16).all(), name
        # frac == 0 exactly at the range ends and on all-zero pixels
        ends = (web == m + 1) | (web == m + D)
        assert np.array_equal(ws[ends], 16 * web[ends]), name
        zero = best == 0
        assert np.array_equal(ws[zero], 16 * (m + D) * np.ones(zero.sum())), name
        assert (web[zero] == m + D).all()
    if D == 1:
        assert np.array_equal(ws, 16 * web)


def test_frac_formula_every_triple():
    """The integer frac against float64 over every (s-, s0, s+) a winner can have with s0 <= 200: s- <= s0, s+ < s0."""
    s0, sm, sp = np.meshgrid(np.arange(201), np.arange(201), np.arange(201), indexing="ij")
    ok = (sm <= s0) & (sp < s0)
    s0, sm, sp = s0[ok], sm[ok], sp[ok]
    den = 2 * s0 - sm - sp
    assert (den >= 1).all()
    got = sub_frac(s0, sm, sp)
    want = np.minimum(7.0, np.floor(16.0 * (sp - sm) / (2.0 * den) + 0.5))
    assert np.array_equal(got, want)
    assert got.min() >= -8 and got.max() <= 7
    assert (got == -8).any() and (got == 7).any()


def test_saturated_maps_sit_on_the_last_shift(orc):
    W, H, D, sw = 24, 16, 6, 5
    z = np.zeros((H, W), np.uint8)
    best, web, ws = match_wta_sub(orc, z, z, D, sw, smb.WRAP, direct=True)
    assert (best == sw * sw).all() and (web == D).all() and (ws == 16 * D).all()
