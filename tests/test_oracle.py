"""CPU tests: pin the oracle (oracle/stereo_oracle.c) before anything trusts it.

 * against tests/golden/golden.json -- CRC32s produced by the UNMODIFIED reference
   (tests/golden/make_golden.py; the fixture rows equal SURVEY.md 8c's table);
 * on the cases compared with the reference itself: against the CRCs stored for them in
   tests/golden/ref_cases.json (tests/ref_cases.py) always, and array for array against
   oracle/_ref (built by oracle/Makefile) when it is present;
 * the fast (separable) box sums against the literal sw*sw tap loop.
"""
import numpy as np
import pytest

import oracle
import ref_cases
from util import FIXTURES, THRESHOLD, load_pair, vname

SURVEY_WEB = {  # SURVEY.md 8(c), the `web` column
    ("1-240x135", 0): "9a354ca2", ("1-240x135", 1): "63ce815c",
    ("2-480x270", 0): "21f7e3d8", ("2-480x270", 1): "dc5c40f5",
    ("3-960x540", 0): "cd445306", ("3-960x540", 1): "7fed09d6",
    ("4-1920x1080", 0): "98dc1e9a", ("4-1920x1080", 1): "c3a8b85c",
    ("5-3840x2160", 0): "824591c4", ("5-3840x2160", 1): "a3363965",
}


def test_golden_matches_survey_table(golden):
    for (name, v), crc in SURVEY_WEB.items():
        assert golden["fixture/%s/%s" % (name, vname(v))]["web"] == crc
    assert golden["synth/c2/wrap"]["web"] == "5b633982"
    assert golden["synth/c2/ghost"]["web"] == "9ef4acd3"


@pytest.mark.parametrize("variant", [oracle.WRAP, oracle.GHOST])
@pytest.mark.parametrize("name", FIXTURES)
def test_oracle_fixture_crcs(orc, golden, name, variant):
    g = golden["fixture/%s/%s" % (name, vname(variant))]
    a, b = load_pair(name)
    assert oracle.crc32(a) == g["left"] and oracle.crc32(b) == g["right"]
    e1, e2 = orc.edges(a, THRESHOLD, variant), orc.edges(b, THRESHOLD, variant)
    assert oracle.crc32(e1) == g["edges1"]
    assert oracle.crc32(e2) == g["edges2"]
    best, web = orc.match_wta(e1, e2, g["D"], g["sw"], variant)
    assert oracle.crc32(best) == g["best"]
    assert oracle.crc32(web) == g["web"]
    assert web.min() >= 1 and web.max() <= g["D"]  # never 0 (SURVEY 3.4)


def test_synth_generator_check_values(orc, golden):
    left, right, disp = orc.synth_pair(1234, 1920, 1080, 64)
    # SURVEY.md 8(d) check values
    assert oracle.crc32(left) == "3c12e05d"
    assert oracle.crc32(right) == "02cda6b6"
    assert oracle.crc32(disp) == "b3f94382"
    assert golden["synth/c2/generator"] == {"left": "3c12e05d", "right": "02cda6b6", "disp": "b3f94382"}


@pytest.mark.parametrize("variant", [oracle.WRAP, oracle.GHOST])
def test_oracle_synth_c2(orc, golden, variant):
    g = golden["synth/c2/%s" % vname(variant)]
    left, right, disp = orc.synth_pair(1234, 1920, 1080, 64)
    e1, e2 = orc.edges(left, THRESHOLD, variant), orc.edges(right, THRESHOLD, variant)
    assert (oracle.crc32(e1), oracle.crc32(e2)) == (g["edges1"], g["edges2"])
    best, web = orc.match_wta(e1, e2, 64, 9, variant)
    assert (oracle.crc32(best), oracle.crc32(web)) == (g["best"], g["web"])
    # known answer (SURVEY 8d): web == d+1 in tile interiors
    D, half, TW, TH = 64, 4, 256, 120
    ys, xs = np.mgrid[0:1080, 0:1920]
    interior = ((xs % TW >= half) & (xs % TW < TW - D - half) & (ys % TH >= half + 1) &
                (ys % TH < TH - half - 1) & (xs >= half + 1) & (xs < 1920 - D - half - 1) &
                (ys >= half + 1) & (ys < 1080 - half - 1))
    agree = (web[interior] == disp[interior] + 1).mean()
    assert agree >= 0.9999, agree


def test_oracle_sweep_crcs(orc, golden):
    a, b = load_pair("1-240x135")
    keys = [k for k in golden if k.startswith("sweep/fix1/")]
    assert len(keys) >= 60
    edges = {v: (orc.edges(a, THRESHOLD, v), orc.edges(b, THRESHOLD, v)) for v in (0, 1)}
    for k in keys:
        g = golden[k]
        v = 1 if g["variant"] == "ghost" else 0
        best, web = orc.match_wta(edges[v][0], edges[v][1], g["D"], g["sw"], v)
        assert (oracle.crc32(best), oracle.crc32(web)) == (g["best"], g["web"]), k
    for k in [k for k in golden if k.startswith("sweep/synth")]:
        g = golden[k]
        v = 1 if g["variant"] == "ghost" else 0
        left, right, _ = orc.synth_pair(77, g["w"], g["h"], g["D"])
        assert oracle.crc32(left) == g["left"]
        e1, e2 = orc.edges(left, THRESHOLD, v), orc.edges(right, THRESHOLD, v)
        assert (oracle.crc32(e1), oracle.crc32(e2)) == (g["edges1"], g["edges2"]), k
        best, web = orc.match_wta(e1, e2, g["D"], g["sw"], v)
        assert (oracle.crc32(best), oracle.crc32(web)) == (g["best"], g["web"]), k


@pytest.mark.parametrize("variant", [oracle.WRAP, oracle.GHOST])
@pytest.mark.parametrize("sw", [1, 2, 3, 8, 21])
def test_fast_box_equals_direct(orc, sw, variant):
    rng = np.random.default_rng(sw * 7 + variant)
    m = (rng.random((37, 53)) < 0.4).astype(np.uint8)
    assert np.array_equal(orc.box(m, sw, variant, True), orc.box(m, sw, variant, False))
    le = (rng.random((37, 53)) < 0.3).astype(np.uint8)
    re = (rng.random((37, 53)) < 0.3).astype(np.uint8)
    bd, wd = orc.match_wta(le, re, 17, sw, variant, direct=True)
    bf, wf = orc.match_wta(le, re, 17, sw, variant, direct=False)
    assert np.array_equal(bd, bf) and np.array_equal(wd, wf)


@pytest.mark.parametrize("variant", [oracle.WRAP, oracle.GHOST])
def test_oracle_equals_reference_build(orc, variant):
    """Array-for-array against the reference's own functions (edges, planes, best, web)."""
    assert ref_cases.build_case(orc, variant) == ref_cases.stored()["build/" + vname(variant)]
    if not oracle.ref_available(variant, 30):
        return  # the live comparison needs the reference built into oracle/_ref
    a, b = load_pair("1-240x135")
    ref = oracle.RefLib(variant, 30)
    e1r, e2r = ref.edges(a, THRESHOLD), ref.edges(b, THRESHOLD)
    e1, e2 = orc.edges(a, THRESHOLD, variant), orc.edges(b, THRESHOLD, variant)
    assert np.array_equal(e1, e1r) and np.array_equal(e2, e2r)
    for sw in (21, 6):
        br, wr, planes = ref.match_wta(e1r, e2r, sw, planes=True)
        bo, wo = orc.match_wta(e1, e2, 30, sw, variant)
        assert np.array_equal(bo, br) and np.array_equal(wo, wr)
        for i in (0, 7, 29):
            m, _, s = orc.shift_planes(e1, e2, sw, i, variant)
            assert np.array_equal(s, planes["scores"][i])
            if variant == oracle.WRAP:
                assert np.array_equal(m, planes["matches"][i])
    # other thresholds move the edge maps; the FP64 order must still agree
    for thr in (0.0, 0.05, 0.5, 1.0):
        assert np.array_equal(orc.edges(a, thr, variant), ref.edges(a, thr))


@pytest.mark.parametrize("variant", [oracle.WRAP, oracle.GHOST])
def test_oracle_equals_reference_other_shift_counts(orc, variant):
    assert ref_cases.shift_counts_case(orc, variant) == ref_cases.stored()["shift_counts/" + vname(variant)]
    for D in ref_cases.SHIFT_COUNTS:
        if not oracle.ref_available(variant, D):
            continue  # the live comparison needs the reference built into oracle/_ref
        left, right = ref_cases.shift_counts_pair(orc, D)
        e1, e2 = orc.edges(left, THRESHOLD, variant), orc.edges(right, THRESHOLD, variant)
        ref = oracle.RefLib(variant, D)
        assert np.array_equal(ref.edges(left, THRESHOLD), e1)
        br, wr = ref.match_wta(e1, e2, 9)
        bo, wo = orc.match_wta(e1, e2, D, 9, variant)
        assert np.array_equal(bo, br) and np.array_equal(wo, wr)


def test_edge_cases(orc):
    # all-equal maps: every shift scores the full window, ties go to the highest shift
    z = np.zeros((30, 40), np.uint8)
    for v in (0, 1):
        best, web = orc.match_wta(z, z, 12, 5, v)
        assert (web == 12).all()
        if v == 0:
            assert (best == 25).all()
        else:
            assert best[0, 0] == 9 and best[15, 20] == 25  # ghost: out-of-image taps add nothing
    # no match anywhere at shift 0 only: left all edges, right none
    o = np.ones((30, 40), np.uint8)
    best, web = orc.match_wta(o, z, 4, 3, 0)
    assert (best == 0).all() and (web == 4).all()  # all-zero column -> num_shifts
    # ghost: right map reads 0 beyond the border, so a 0-valued left pixel matches there
    best, web = orc.match_wta(o, o, 4, 1, 1)
    assert best[0, 0] == 1 and web[0, 39] == 1 and web[0, 0] == 4


def test_step3(orc):
    a, b = load_pair("1-240x135")
    e1, e2 = orc.edges(a, THRESHOLD, 0), orc.edges(b, THRESHOLD, 0)
    _, web = orc.match_wta(e1, e2, 30, 21, 0)
    filled = orc.fill_web_holes(web, 32)
    assert np.array_equal(filled, web)  # provable no-op (SURVEY 3.4)
    rc, out = orc.draw_contour_map(filled, 10)
    assert rc == 0
    mn, mx = web.min(), web.max()
    assert np.array_equal(out, (((web - mn) % ((mx - mn) // 10)) == 0).astype(np.uint8))
    rc, _ = orc.draw_contour_map(np.full((4, 4), 7, np.int32), 10)
    assert rc == 1  # degenerate: the reference would divide by zero
    holes = web.copy()
    holes[10:12, 10:12] = 0
    f2 = orc.fill_web_holes(holes, 3)
    assert f2.shape == web.shape


def test_fill_web_holes_equals_reference(orc):
    """Holes (zeros) at row ends: the reference's unwrapped IDX(x+-1, y) makes the last pixel of a row a neighbour
    of the first pixel of the next (stereo.c:237-243).  Holes stay away from the first and last rows, where the
    reference reads outside the array; an even number of passes, so that it returns (and does not free) our buffer."""
    assert ref_cases.fill_holes_case(orc) == ref_cases.stored()["fill_web_holes"]
    if not oracle.ref_available(oracle.WRAP, 30):
        return  # the live comparison needs the reference built into oracle/_ref
    import ctypes as C
    web = ref_cases.holes_web()
    h, w = web.shape
    L = oracle.RefLib(oracle.WRAP, 30).L
    L.fill_web_holes.restype = C.c_void_p
    for times in ref_cases.HOLE_PASSES:
        ref = np.ascontiguousarray(web.copy())
        p = L.fill_web_holes(ref.ctypes.data_as(C.c_void_p), w, h, times)
        assert p == ref.ctypes.data
        assert np.array_equal(orc.fill_web_holes(web, times), ref), times


@pytest.mark.parametrize("variant", [oracle.WRAP, oracle.GHOST])
def test_oracle_equals_reference_wide_windows(orc, variant):
    """Windows beyond the reference default (23..63): the GPU tests use the oracle as checker there too, so the
    oracle is pinned to the reference's own functions for them (small frames: the reference does sw*sw taps)."""
    assert ref_cases.wide_windows_case(orc, variant) == ref_cases.stored()["wide_windows/" + vname(variant)]
    for (w, h, D, sw) in ref_cases.WIDE_WINDOWS:
        if not oracle.ref_available(variant, D):
            continue  # the live comparison needs the reference built into oracle/_ref
        le, re = ref_cases.wide_windows_maps(w, h, sw)
        br, wr = oracle.RefLib(variant, D).match_wta(le, re, sw)
        bo, wo = orc.match_wta(le, re, D, sw, variant)
        assert np.array_equal(bo, br) and np.array_equal(wo, wr), (w, h, D, sw)
