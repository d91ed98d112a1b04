"""The float64 model of the edge detector (tests/edge_model.py) and its probe images, on the CPU.

The model is pinned to the oracle here, and the oracle is pinned to the reference (test_oracle.py); the GPU edge
tests (test_gpu_edges.py) then compare the library with the oracle on the probe images built here.
"""
import numpy as np
import pytest

import edge_model as em
from util import FIXTURES, THRESHOLD, load_pair, vname

# Boundary pairs (A, B) no stencil can put in front of one detector while the other three stay silent, the same for
# every direction.  Near 0 any difference fires: (0, 1) needs the other three detectors to compare equal sums, which
# forces every cell of the larger sum to 0; (764, 765) likewise forces every cell to 255.  Every other boundary entry
# of every tested threshold has a decisive stencil.
INFEASIBLE = {0.0: {(0, 1), (1, 0), (764, 765), (765, 764)},
              5e-324: {(0, 1), (1, 0), (764, 765), (765, 764)},
              1e-4: {(0, 1), (1, 0), (764, 765), (765, 764)},
              2.5e-3: {(0, 1), (1, 0)}}

W_PROBE, H_PROBE = 256, 120


def thr_id(t):
    return "%.4g" % t


@pytest.mark.parametrize("variant", [em.WRAP, em.GHOST], ids=vname)
@pytest.mark.parametrize("thr", em.THRESHOLDS, ids=thr_id)
def test_model_equals_oracle_on_probe_frames(orc, thr, variant):
    frames, _ = em.probe_frames(thr, variant, W_PROBE, H_PROBE)
    for f in frames:
        assert np.array_equal(em.model_edges(f, thr, variant), orc.edges(f, thr, variant))
    # and on a generic width with a frame seam through a probe column
    frames, _ = em.probe_frames(thr, variant, 37, 40)
    for f in frames[:4]:
        assert np.array_equal(em.model_edges(f, thr, variant), orc.edges(f, thr, variant))


@pytest.mark.parametrize("variant", [em.WRAP, em.GHOST], ids=vname)
def test_model_equals_oracle_on_fixtures(orc, variant):
    for name in FIXTURES:
        for img in load_pair(name):
            assert np.array_equal(em.model_edges(img, THRESHOLD, variant), orc.edges(img, THRESHOLD, variant)), name


@pytest.mark.parametrize("thr", em.THRESHOLDS, ids=thr_id)
def test_table_is_symmetric_and_monotone(thr):
    """edge(L, R) == max(L, R) > hi[min(L, R)] exactly, for every pair of sums.  This is why k_edge_thresholds
    leaves its flag at 1 (INFO_EDGE_THRESHOLDS reads 1) for every threshold in [0, 1], which is all the ABI accepts:
    the bit-table fallback of the detector kernels (edge_lut) cannot be reached from the ABI, so no test runs it."""
    t, h = em.detect_table(thr), em.hi(thr)
    assert np.array_equal(t, t.T)
    s = np.arange(em.NSUM)
    mn, mx = np.minimum(s[:, None], s[None, :]), np.maximum(s[:, None], s[None, :])
    assert np.array_equal(t, mx > h[mn])
    assert (h >= s).all()  # no edge at L == R


@pytest.mark.parametrize("thr", em.THRESHOLDS, ids=thr_id)
def test_probes_cover_every_boundary_entry(thr):
    """Every ordered boundary pair (both orders of (m, hi[m]) and (m, hi[m] + 1)) sits decisively in front of each of
    the four detectors somewhere in the probe frames of both variants, apart from the recorded infeasible pairs."""
    bp = set(map(tuple, em.boundary_pairs(thr).tolist()))
    assert len(bp) > 1000
    infeasible = INFEASIBLE.get(thr, set())
    for variant in (em.WRAP, em.GHOST):
        frames, _ = em.probe_frames(thr, variant, W_PROBE, H_PROBE)
        hits = [set() for _ in range(4)]
        for f in frames:
            for d, s in enumerate(em.decisive_hits(f, thr, variant)):
                hits[d] |= s
        for d in range(4):
            assert hits[d] <= bp
            assert bp - hits[d] == infeasible, (em.DIRECTIONS[d], variant, sorted(bp - hits[d])[:8])
            for order in (np.less, np.greater, np.equal):  # A < B, A > B and, where hi[m] == m, A == B
                want = {p for p in bp - infeasible if order(*p)}
                assert {p for p in hits[d] if order(*p)} == want


def test_probe_placement_covers_word_lanes_and_seams():
    """Probe centres run through every residue of x mod 4 (a thread's nibble) and mod 32 (the shuffled word); WRAP
    frames have probes centred on all four seams, GHOST frames none on the border."""
    for variant in (em.WRAP, em.GHOST):
        _, where = em.probe_frames(0.15, variant, W_PROBE, H_PROBE)
        xs = {x for w in where for x, _ in w}
        ys = {y for w in where for _, y in w}
        assert {x % 32 for x in xs} == set(range(32))
        if variant == em.WRAP:
            assert {0, W_PROBE - 1} <= xs and {0, H_PROBE - 1} <= ys
        else:
            assert min(xs) >= 1 and max(xs) <= W_PROBE - 2 and min(ys) >= 1 and max(ys) <= H_PROBE - 2
