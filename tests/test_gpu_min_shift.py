"""Search ranges that start above zero (sm_create_range and its band / multi / bands twins) on the GPU.

A context with min_shift m and num_shifts D searches the shifts [m, m + D).  The expected values are numpy's
winner-take-all over the oracle's score planes oracle.shift_planes(le, re, sw, s, variant) for s in [m, m + D) --
ties to the highest shift, all-zero pixels at web = m + D -- on the oracle's edge maps.  Covered: both variants, the
bit-sliced and the direct kernel, every bit-sliced shape family (asserted through SM_INFO_KERNEL_SHAPE), minimum
shifts around the word, chunk and frame widths, odd frame sizes and widths that are no multiple of 4 (the producers'
generic kernels), every entry from the edge detector to the batch pipelines, band / multi / bands objects, the debug
planes, guard values, the m = 0 goldens, two full-size frames and a seeded random sample."""
import os
import subprocess
import zlib

import numpy as np
import pytest

import oracle
import stereomatching_b200 as smb
from test_gpu_flavours import FLAVOURS, code, diff, families, run_dev_batch
from test_gpu_web16 import run16
from util import ROOT, THRESHOLD, load_pair, vname

pytestmark = pytest.mark.gpu

VARIANTS = [smb.WRAP, smb.GHOST]
KERNELS = {smb.KERNEL_AUTO: "auto", smb.KERNEL_DIRECT: "direct"}


@pytest.fixture(scope="module")
def num_sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def m_values(W):
    return [1, 3, 4, 31, 32, 33, 64, 100, W - 1, W, 2 * W + 3]


def expected(orc, le, re, m, D, sw, variant):
    """(best, web) of the range [m, m + D): the oracle's score planes, winner-take-all in numpy."""
    H, W = le.shape
    best = np.zeros((H, W), np.int32)
    web = np.zeros((H, W), np.int32)
    for s in range(m, m + D):
        score = orc.shift_planes(le, re, sw, s, variant)[2]
        take = score >= best
        best = np.where(take, score, best)
        web = np.where(take, s + 1, web)
    return best, web


def check(best, web, bo, wo, what):
    assert np.array_equal(web, wo), "%s: web %s" % (what, diff(web, wo))
    assert np.array_equal(best, bo), "%s: best %s" % (what, diff(best, bo))


def image_pair(orc, seed, W, H, m, D):
    """8-bit pair whose second image is the first shifted by m + the synthetic disparity in [0, D) (SURVEY 8d)."""
    left, _, disp = orc.synth_pair(seed, W, H, D)
    xs = (np.arange(W)[None, :] - m - disp) % W
    right = np.ascontiguousarray(np.take_along_axis(left, xs, axis=1))
    return left, right, disp


# ---------------------------------------------------------------------------------
# the hot kernels: every bit-sliced shape family and the direct kernel, packed by k_pack
# ---------------------------------------------------------------------------------
@pytest.mark.parametrize("kernel", list(KERNELS), ids=KERNELS.get)
@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
@pytest.mark.parametrize("flavour", list(FLAVOURS))
def test_shape_family(orc, num_sms, flavour, variant, kernel):
    nw, seg, multi, c2, hp, halves, geometry = FLAVOURS[flavour]
    half = halves[len(halves) // 2]
    W, H1, Hn, D = geometry(half, num_sms)
    sw = 2 * half + 1
    want = code(half, nw, seg, c2, hp, multi) if kernel == smb.KERNEL_AUTO else smb.SHAPE_DIRECT
    one_pair = H1 <= 64  # (the one-word kernel's one-pair geometry has a CTA per SM: its batch geometry covers it)
    for m in m_values(W):
        tag = "%s half %d W %d D %d m %d %s %s" % (flavour, half, W, D, m, vname(variant), KERNELS[kernel])
        if one_pair:
            fams = families(W, H1, D, 31 * m + W)
            with smb.StereoContext(W, H1, D, sw, variant, kernel=kernel, min_shift=m) as c:
                for name, le, re in (fams[0], fams[1], fams[3]):  # two random densities, never-matching maps
                    best, web = c.match_wta_host(le, re)
                    assert c.get_info(smb.INFO_KERNEL_SHAPE) == want, tag
                    check(best, web, *expected(orc, le, re, m, D, sw, variant), "%s %s" % (tag, name))
        if Hn is not None:
            rng = np.random.default_rng(m * 7 + D)
            les = [(rng.random((Hn, W)) < p).astype(np.uint8) for p in (0.2, 0.5)]
            res = [(rng.random((Hn, W)) < p).astype(np.uint8) for p in (0.3, 0.5)]
            with smb.StereoContext(W, Hn, D, sw, variant, kernel=kernel, min_shift=m) as c:
                best, web = run_dev_batch(c, les, res)
                assert c.get_info(smb.INFO_KERNEL_SHAPE) == want, tag
                for k in range(2):
                    check(best[k], web[k], *expected(orc, les[k], res[k], m, D, sw, variant), "%s pair %d" % (tag, k))


# ---------------------------------------------------------------------------------
# the producers: edges straight into the planes (word path, funnel offsets, generic kernels), the FP64 detector,
# the byte maps, the debug planes and the narrowed webs
# ---------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
@pytest.mark.parametrize("W,H", [(128, 40), (96, 33), (67, 29), (130, 21)])
def test_edges_entries(orc, variant, W, H):
    D, sw = 24, 7
    for m in m_values(W):
        tag = "%dx%d m %d %s" % (W, H, m, vname(variant))
        left, right, _ = image_pair(orc, 7 * m + W, W, H, m, D)
        e1, e2 = orc.edges(left, THRESHOLD, variant), orc.edges(right, THRESHOLD, variant)
        bo, wo = expected(orc, e1, e2, m, D, sw, variant)
        with smb.StereoContext(W, H, D, sw, variant, min_shift=m) as c:
            c.upload_u8(left, right)
            c.edges(THRESHOLD)
            assert np.array_equal(c.download(smb.EDGES1), e1), tag
            assert np.array_equal(c.download(smb.EDGES2), e2), tag  # the whole second map, unshifted
            c.match_wta()
            check(c.download(smb.BEST), c.download(smb.WEB), bo, wo, tag)
            # debug planes at real shifts inside the range, rejection outside it
            for s in (m, m + 5, m + D - 1):
                mo, ao, so = orc.shift_planes(e1, e2, sw, s, variant)
                assert np.array_equal(c.download(smb.MATCH, s), mo), (tag, s)
                assert np.array_equal(c.download(smb.SCORE_ALL, s), ao), (tag, s)
                assert np.array_equal(c.download(smb.SCORE, s), so), (tag, s)
            for s in (m - 1, m + D, -1):
                with pytest.raises(smb.StereoError) as e:
                    c.download(smb.SCORE, s)
                assert e.value.code == -1
            assert np.array_equal(c.download_web_u16(), wo.astype(np.uint16)), tag
            if m + D <= 255:
                assert np.array_equal(c.download_web_u8(), wo.astype(np.uint8)), tag
            else:
                with pytest.raises(smb.StereoError):
                    c.download_web_u8()
            # step 3 on a range web: web >= m + 1 everywhere, so hole filling is the identity
            c.fill_web_holes(4)
            assert np.array_equal(c.download(smb.WEB_FILLED), wo), tag
            # the FP64 detector and the byte maps packed by k_pack
            c.set_option(smb.OPT_EDGES_FP64, 1)
            c.edges(THRESHOLD)
            assert np.array_equal(c.download(smb.EDGES2), e2), tag
            c.match_wta()
            check(c.download(smb.BEST), c.download(smb.WEB), bo, wo, tag + " fp64")


@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
@pytest.mark.parametrize("W,H", [(128, 36), (67, 29)])
def test_run_batch(orc, variant, W, H):
    D, sw, n = 40, 9, 5
    for m in (3, 33, W + 5, 300):
        tag = "%dx%d m %d %s" % (W, H, m, vname(variant))
        pairs = [image_pair(orc, 1234 + 2 * k + m, W, H, m, D) for k in range(n)]
        first = np.stack([p[0] for p in pairs])
        second = np.stack([p[1] for p in pairs])
        want = [expected(orc, orc.edges(p[0], THRESHOLD, variant), orc.edges(p[1], THRESHOLD, variant), m, D, sw,
                         variant) for p in pairs]
        bo = np.stack([w[0] for w in want])
        wo = np.stack([w[1] for w in want])
        with smb.StereoContext(W, H, D, sw, variant, min_shift=m) as c:
            c.set_option(smb.OPT_PIPE_GROUP, 2)  # several stages, a ragged last one
            web, best = c.run_batch(first, second, THRESHOLD, want_best=True)
            check(best, web, bo, wo, tag + " i32")
            web16, best16 = c.run_batch(first, second, THRESHOLD, want_best=True, web16=True)
            check(best16.astype(np.int32), web16.astype(np.int32), bo, wo, tag + " u16")
            if m + D <= 255:
                assert np.array_equal(c.run_batch(first, second, THRESHOLD, web_u8=True), wo.astype(np.uint8)), tag
            else:
                with pytest.raises(smb.StereoError):
                    c.run_batch(first, second, THRESHOLD, web_u8=True)
        with smb.MultiGpuBatch([0, 0], W, H, D, sw, variant, min_shift=m) as mb:
            web, best = mb.run_batch(first, second, THRESHOLD, want_best=True)
            check(best, web, bo, wo, tag + " multi i32")
            assert np.array_equal(mb.run_batch(first, second, THRESHOLD, web16=True), wo.astype(np.uint16)), tag


@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
def test_dev_batch_ragged_with_guards(orc, variant):
    """17 pairs (a ragged last launch) through sm_match_wta_dev_batch and ..16 with and without best; the 16-bit
    outputs sit between 0xFFFF guards that must survive."""
    W, H, D, sw, m = 64, 24, 40, 9, 37
    rng = np.random.default_rng(5)
    les = [(rng.random((H, W)) < 0.3).astype(np.uint8) for _ in range(17)]
    res = [np.roll(le, m + int(rng.integers(0, D)), axis=1) ^ (rng.random((H, W)) < 0.05).astype(np.uint8)
           for le in les]
    want = [expected(orc, le, re, m, D, sw, variant) for le, re in zip(les, res)]
    with smb.StereoContext(W, H, D, sw, variant, min_shift=m) as c:
        best, web = run_dev_batch(c, les, res)
        for k in range(17):
            check(best[k], web[k], *want[k], "i32 pair %d" % k)
        for with_best in (True, False):
            b16, w16 = run16(c, les, res, with_best=with_best)
            for k in range(17):
                assert np.array_equal(w16[k], want[k][1]), ("u16 web", with_best, k)
                if with_best:
                    assert np.array_equal(b16[k], want[k][0]), ("u16 best", k)


# ---------------------------------------------------------------------------------
# band contexts, sm_multi_* and sm_bands_*
# ---------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
def test_bands(orc, variant):
    W, H, D, sw = 96, 45, 30, 9
    for m in (35, 97):
        left, right, _ = image_pair(orc, 99 + m, W, H, m, D)
        bo, wo = expected(orc, orc.edges(left, THRESHOLD, variant), orc.edges(right, THRESHOLD, variant), m, D, sw,
                          variant)
        web = np.full((H, W), -1, np.int32)
        best = np.full((H, W), -1, np.int32)
        for r0, r1 in ((0, 13), (13, 20), (20, H)):
            with smb.StereoContext(W, H, D, sw, variant, rows=(r0, r1), min_shift=m) as c:
                c.upload_u8(left, right)
                c.edges(THRESHOLD)
                c.match_wta()
                c.download(smb.WEB, out=web)
                c.download(smb.BEST, out=best)
        check(best, web, bo, wo, "bands m %d" % m)
        with smb.MultiGpuBands([0, 0], W, H, D, sw, variant, min_shift=m) as mb:
            web, best = mb.run(left, right, THRESHOLD, want_best=True)
            check(best, web, bo, wo, "sm_bands m %d" % m)
            web16, best16 = mb.run(left, right, THRESHOLD, want_best=True, web16=True)
            check(best16.astype(np.int32), web16.astype(np.int32), bo, wo, "sm_bands16 m %d" % m)


# ---------------------------------------------------------------------------------
# min_shift = 0 through the range creators: the reference's goldens
# ---------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
@pytest.mark.parametrize("fixture", ["1-240x135", "2-480x270"])
def test_zero_range_is_the_reference(golden, fixture, variant):
    g = golden["fixture/%s/%s" % (fixture, vname(variant))]
    left, right = load_pair(fixture)
    W, H, D, sw = g["w"], g["h"], g["D"], g["sw"]
    # sm_create_range itself, under the binding's context methods
    h = smb.api.C.c_void_p()
    smb.api._check(smb.lib().sm_create_range(smb.api.C.byref(h), 0, W, H, 0, D, sw, variant))
    c = smb.StereoContext.__new__(smb.StereoContext)
    c.W, c.H, c.D, c.sw, c.variant, c.min_shift, c.row0, c.row1, c._c = W, H, D, sw, variant, 0, 0, H, h
    with c:
        c.upload_u8(left, right)
        c.edges(g["threshold"])
        c.match_wta()
        assert oracle.crc32(c.download(smb.WEB)) == g["web"]
        assert oracle.crc32(c.download(smb.BEST)) == g["best"]
    with smb.MultiGpuBands([0, 0], W, H, D, sw, variant, min_shift=0) as mb:
        web, best = mb.run(left, right, g["threshold"], want_best=True)
        assert (oracle.crc32(web), oracle.crc32(best)) == (g["web"], g["best"])
    with smb.MultiGpuBatch([0, 0], W, H, D, sw, variant, min_shift=0) as mb:
        web = mb.run_batch(left[None], right[None], g["threshold"])
        assert oracle.crc32(web[0]) == g["web"]


# ---------------------------------------------------------------------------------
# full size, without the oracle
# ---------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
def test_1080p_fixture_range_is_a_slice_of_the_score_planes(golden, variant):
    """(m, D) = (20, 30) on the 1080p fixture equals the winner-take-all over SM_SCORE planes 20..49 of a (0, 50)
    context."""
    name = "4-1920x1080"
    g = golden["fixture/%s/%s" % (name, vname(variant))]
    left, right = load_pair(name)
    W, H, sw = g["w"], g["h"], g["sw"]
    with smb.StereoContext(W, H, 50, sw, variant) as c:
        c.upload_u8(left, right)
        c.edges(THRESHOLD)
        bo = np.zeros((H, W), np.int32)
        wo = np.zeros((H, W), np.int32)
        for s in range(20, 50):
            score = c.download(smb.SCORE, s)
            take = score >= bo
            bo = np.where(take, score, bo)
            wo = np.where(take, s + 1, wo)
    with smb.StereoContext(W, H, 30, sw, variant, min_shift=20) as c:
        c.upload_u8(left, right)
        c.edges(THRESHOLD)
        c.match_wta()
        check(c.download(smb.BEST), c.download(smb.WEB), bo, wo, "1080p fixture (20, 30)")


@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
def test_1080p_band_96_160_known_answer(orc, variant):
    """A synthetic 1080p pair with disparities in [96, 160), searched at (96, 64): web == d + 1 in the tile interiors
    (SURVEY 8d) for at least 99.99 % of the pixels."""
    W, H, m, D, sw = 1920, 1080, 96, 64, 9
    left, right, disp = image_pair(orc, 1234, W, H, m, D)
    half = sw // 2
    tw, th = max(240, 4 * D), 120
    with smb.StereoContext(W, H, D, sw, variant, min_shift=m) as c:
        c.upload_u8(left, right)
        c.edges(THRESHOLD)
        c.match_wta()
        web = c.download(smb.WEB)
        assert c.get_info(smb.INFO_KERNEL_SHAPE) == code(half, 2, 16)
        web16 = c.run_batch(left[None], right[None], THRESHOLD, web16=True)[0]
    assert np.array_equal(web16, web.astype(np.uint16))
    ys, xs = np.mgrid[0:H, 0:W]
    interior = ((xs % tw >= half) & (xs % tw < tw - m - D - half) & (ys % th >= half + 1) & (ys % th < th - half - 1) &
                (xs >= half) & (xs < W - m - D - half) & (ys >= half + 1) & (ys < H - half - 1))
    agree = (web[interior] == m + disp[interior] + 1).mean()
    assert agree >= 0.9999, agree


# ---------------------------------------------------------------------------------
# a seeded random sample
# ---------------------------------------------------------------------------------
def test_random_sample(orc):
    rng = np.random.default_rng(20261021)
    for case in range(40):
        W, H = int(rng.integers(9, 200)), int(rng.integers(5, 60))
        sw = int(rng.integers(0, min(W, H, 25) + 1))
        D = int(rng.choice([int(rng.integers(1, 17)), int(rng.integers(17, 65)), int(rng.integers(65, 140))]))
        m = int(rng.integers(0, 3 * W + 40))
        variant = int(rng.integers(0, 2))
        tag = "case %d: %dx%d sw %d m %d D %d %s" % (case, W, H, sw, m, D, vname(variant))
        le = (rng.random((H, W)) < rng.uniform(0.1, 0.7)).astype(np.uint8)
        re = np.roll(le, m + int(rng.integers(0, D)), axis=1) ^ (rng.random((H, W)) < 0.05).astype(np.uint8)
        with smb.StereoContext(W, H, D, sw, variant, min_shift=m) as c:
            best, web = c.match_wta_host(le, re)
        check(best, web, *expected(orc, le, re, m, D, sw, variant), tag)


# ---------------------------------------------------------------------------------
# stereobatch's trailing min_shift
# ---------------------------------------------------------------------------------
def test_stereobatch_min_shift(orc):
    exe = os.path.join(ROOT, "timing", "stereobatch")
    W, H, D, sw, n = 96, 40, 24, 7, 3

    def crc(*extra):
        out = subprocess.run([exe, str(W), str(H), str(D), str(sw), str(n), "wrap", "i32", *extra],
                             capture_output=True, text=True, check=True).stdout
        return out.strip().split("web_crc32 = ")[1]

    assert crc("1", "0") == crc("1")  # min_shift 0 is the run without one
    m = 45
    pairs = [image_pair(orc, 1234 + 2 * k, W, H, m, D) for k in range(n)]
    with smb.StereoContext(W, H, D, sw, smb.WRAP, min_shift=m) as c:
        web = c.run_batch(np.stack([p[0] for p in pairs]), np.stack([p[1] for p in pairs]), THRESHOLD)
    assert crc("1", str(m)) == "%08x" % zlib.crc32(web.tobytes())
