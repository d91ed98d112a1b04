"""The edge detector (step 1) on the GPU against the oracle, at every boundary of its threshold table.

Every result of the library starts with the edges, and the 8-bit detector decides them with integer thresholds
derived from a table of the reference's FP64 expression (k_edges.cu).  The probe frames of tests/edge_model.py put
every boundary entry of a threshold's table in front of one detector of one pixel while the other three stay silent,
so that one wrong threshold, table bit or stencil cell changes an edge bit.  Here the library's detectors see them:
  * the byte maps of sm_edges (k_edges_planes with WRITE_U8), at regular widths (the word path) and the others (the
    gathering kernels), in whole frames and band contexts;
  * the same frames with SM_OPT_EDGES_FP64 (k_edges<uint8_t>) and through sm_upload_f64 (k_edges<double>);
  * the planes alone (k_edges_planes without WRITE_U8), read pixel-exact through sm_run_batch, sm_run_batch16 and
    sm_multi_run_batch at one shift and a one-pixel window, where best is 1 exactly where the two edge bits agree;
  * halo rows of bands, through band contexts and sm_bands_run;
  * the GHOST border rule, and a switch of threshold between every kind of call on one context.
"""
import functools

import numpy as np
import pytest

import edge_model as em
import stereomatching_b200 as smb
from util import vname

pytestmark = pytest.mark.gpu

THRS = em.THRESHOLDS


def thr_id(t):
    return "%.4g" % t


@functools.lru_cache(maxsize=None)
def _frames(thr, variant, w, h):
    return em.probe_frames(thr, variant, w, h)[0]


def _load(c, a, b, src):
    """src: "u8" (k_edges_planes), "fp64" (SM_OPT_EDGES_FP64: k_edges<uint8_t>) or "f64" (k_edges<double>)."""
    if src == "f64":
        c.upload_f64(a / 256.0, b / 256.0)
    else:
        c.set_option(smb.OPT_EDGES_FP64, int(src == "fp64"))
        c.upload_u8(a, b)


def _check_edges(orc, c, a, b, thr, variant, src, rows=None):
    c.edges(thr)
    if src == "u8":
        assert c.get_info(smb.INFO_EDGE_THRESHOLDS) == 1
    h, w = a.shape
    r0, r1 = rows if rows else (0, h)
    for which, img in ((smb.EDGES1, a), (smb.EDGES2, b)):
        got = np.full((h, w), 7, np.uint8)
        c.download(which, out=got)
        want = orc.edges(img, thr, variant)
        assert np.array_equal(got[r0:r1], want[r0:r1]), (which, np.argwhere(got[r0:r1] != want[r0:r1])[:5])


SOURCES = ["u8", "fp64", "f64"]
# width -> frame height: W = 4 (a thread's neighbouring words are its own, through the torus), 36 (a last word that is
# partly padding), 256; and widths = 1, 2, 3 mod 4 (the gathering kernels)
WIDTHS = {4: 3000, 36: 300, 256: 120, 37: 300, 38: 300, 39: 300}


@pytest.mark.parametrize("src", SOURCES)
@pytest.mark.parametrize("variant", [smb.WRAP, smb.GHOST], ids=vname)
@pytest.mark.parametrize("thr", THRS, ids=thr_id)
def test_edge_maps_whole_frames(orc, thr, variant, src):
    for w, h in WIDTHS.items():
        fr = _frames(thr, variant, w, h)
        with smb.StereoContext(w, h, 1, 1, variant) as c:
            for i in range(len(fr)):
                a, b = fr[i], fr[(i + 1) % len(fr)][::-1]
                _load(c, a, b, src)
                _check_edges(orc, c, a, b, thr, variant, src)


def _small_frame(rng, w, h):
    """Random content with small steps (ties and near-ties of neighbouring sums) and some jumps."""
    walk = np.cumsum(rng.integers(-3, 4, (h, w)), axis=1) + rng.integers(0, 256, (h, 1))
    img = np.where(rng.random((h, w)) < 0.15, rng.integers(0, 256, (h, w)), walk)
    return np.clip(img, 0, 255).astype(np.uint8)


SMALL = [(256, 2), (36, 3), (4, 2), (37, 2), (38, 3), (39, 3), (2, 2), (3, 3), (1, 64), (64, 1), (1, 1), (1, 3)]


@pytest.mark.parametrize("src", SOURCES)
@pytest.mark.parametrize("variant", [smb.WRAP, smb.GHOST], ids=vname)
@pytest.mark.parametrize("thr", THRS, ids=thr_id)
def test_edge_maps_small_frames(orc, thr, variant, src):
    """Frames of two and three rows (a stencil's rows wrap onto each other / both touch the ghost rows) and one-pixel
    wide or high frames."""
    rng = np.random.default_rng(5)
    for w, h in SMALL:
        with smb.StereoContext(w, h, 1, 1, variant) as c:
            for _ in range(3):
                a, b = _small_frame(rng, w, h), _small_frame(rng, w, h)
                _load(c, a, b, src)
                _check_edges(orc, c, a, b, thr, variant, src)


@pytest.mark.parametrize("src", SOURCES)
@pytest.mark.parametrize("variant", [smb.WRAP, smb.GHOST], ids=vname)
@pytest.mark.parametrize("thr", THRS, ids=thr_id)
def test_edge_maps_band_contexts(orc, thr, variant, src):
    """Band contexts: 2 and 3 bands of a probe frame, and 3-row bands of a 21-row frame with a 21-pixel window,
    whose padded rows (band + 2 * half) exceed the frame: they repeat (WRAP) or reach outside it on both sides
    (GHOST), and the FP64 kernels cover the whole frame."""
    cases = [(36, 150, 21, (2, 3)), (37, 150, 21, (2, 3)), (36, 21, 21, (7,)), (39, 21, 21, (7,))]
    for w, h, sw, bands in cases:
        fr = _frames(thr, variant, w, h)
        a, b = fr[0], fr[-1][:, ::-1]
        for n in bands:
            for k in range(n):
                rows = smb.band_rows(h, n, k)
                with smb.StereoContext(w, h, 1, sw, variant, rows=rows) as c:
                    _load(c, a, b, src)
                    _check_edges(orc, c, a, b, thr, variant, src, rows=rows)


# ---- the planes alone: best at one shift and a one-pixel window is [edge1 == edge2] -------------------------------
def _plane_pairs(thr, variant, w, h):
    """(probe, flat) pairs read the first image's planes LA / LB, (flat, probe) pairs the second's RB.  At least 17
    pairs and a count that is no multiple of the pipeline's group of 3: the buffer sets rotate, the last group is
    ragged."""
    fr = list(_frames(thr, variant, w, h))
    flat = np.full((h, w), 100, np.uint8)
    pairs = [(p, flat) for p in fr] + [(flat, p) for p in fr]
    k = 0
    while len(pairs) < 17 or len(pairs) % 3 == 0:
        pairs.append((fr[k % len(fr)], fr[(k + 1) % len(fr)][::-1]))
        k += 1
    return np.stack([p[0] for p in pairs]), np.stack([p[1] for p in pairs])


def _want(orc, first, second, thr, variant, num_shifts=1, sw=1):
    out = [orc.match_wta(orc.edges(a, thr, variant), orc.edges(b, thr, variant), num_shifts, sw, variant)
           for a, b in zip(first, second)]
    return np.stack([o[0] for o in out]), np.stack([o[1] for o in out])


def _devices(n):
    ndev = smb.device_count()
    return [k % ndev for k in range(n)]


# (256, 24): the word path; (255, 25): an odd width, and pair k's image base is unaligned for odd k (GENERIC kernels)
PLANE_SIZES = [(256, 24), (255, 25)]


@pytest.mark.parametrize("variant", [smb.WRAP, smb.GHOST], ids=vname)
@pytest.mark.parametrize("thr", THRS, ids=thr_id)
def test_planes_through_run_batch(orc, thr, variant):
    for w, h in PLANE_SIZES:
        first, second = _plane_pairs(thr, variant, w, h)
        bo, wo = _want(orc, first, second, thr, variant)
        with smb.StereoContext(w, h, 1, 1, variant) as c:
            c.set_option(smb.OPT_PIPE_GROUP, 3)
            web, best = c.run_batch(first, second, thr, want_best=True)
            assert np.array_equal(best, bo) and np.array_equal(web, wo), (w, h)
            assert c.get_info(smb.INFO_EDGE_THRESHOLDS) == 1
            web, best = c.run_batch(first, second, thr, web_u8=True, want_best=True)
            assert np.array_equal(best, bo) and np.array_equal(web, wo.astype(np.uint8)), (w, h)
            web, best = c.run_batch(first, second, thr, want_best=True, web16=True)
            assert np.array_equal(best, bo.astype(np.uint16)) and np.array_equal(web, wo.astype(np.uint16)), (w, h)
        with smb.MultiGpuBatch(_devices(3), w, h, 1, 1, variant) as m:
            web, best = m.run_batch(first, second, thr, want_best=True)
            assert np.array_equal(best, bo) and np.array_equal(web, wo), (w, h)
            web, best = m.run_batch(first, second, thr, want_best=True, web16=True)
            assert np.array_equal(best, bo.astype(np.uint16)), (w, h)


@pytest.mark.parametrize("variant", [smb.WRAP, smb.GHOST], ids=vname)
@pytest.mark.parametrize("thr", THRS, ids=thr_id)
def test_planes_through_run_batch_fp64(orc, thr, variant):
    """sm_run_batch with SM_OPT_EDGES_FP64: k_edges<uint8_t> per image of every group, then k_pack."""
    for w, h in PLANE_SIZES:
        first, second = _plane_pairs(thr, variant, w, h)
        bo, wo = _want(orc, first, second, thr, variant)
        with smb.StereoContext(w, h, 1, 1, variant) as c:
            c.set_option(smb.OPT_PIPE_GROUP, 3)
            c.set_option(smb.OPT_EDGES_FP64, 1)
            web, best = c.run_batch(first, second, thr, want_best=True)
            assert np.array_equal(best, bo) and np.array_equal(web, wo), (w, h)
            web, best = c.run_batch(first, second, thr, want_best=True, web16=True)
            assert np.array_equal(best, bo.astype(np.uint16)), (w, h)


# ---- halo rows: a band's edges reach half rows beyond its own ------------------------------------------------------
def _bands_check(orc, w, h, sw, n, a, b, thr, variant, bo, wo):
    best = np.full((h, w), -1, np.int32)
    web = np.full((h, w), -1, np.int32)
    for k in range(n):
        with smb.StereoContext(w, h, 1, sw, variant, rows=smb.band_rows(h, n, k)) as c:
            c.upload_u8(a, b)
            c.edges(thr)
            c.match_wta()
            c.download(smb.BEST, out=best)
            c.download(smb.WEB, out=web)
    assert np.array_equal(best, bo) and np.array_equal(web, wo), (w, h, sw, n)


@pytest.mark.parametrize("variant", [smb.WRAP, smb.GHOST], ids=vname)
@pytest.mark.parametrize("thr", THRS, ids=thr_id)
def test_halo_rows(orc, thr, variant):
    """One shift, a 3 x 3 window: best counts the agreeing edge bits around each pixel, so one wrong edge bit of a
    halo row changes best in the band beside it.  Band contexts and sm_bands_run over 2 and 3 slots; and 3-row bands
    of a 21-row frame with a 21-pixel window, where band + 2 * half exceeds the frame."""
    for w, h, sw, counts in [(256, 120, 3, (2, 3)), (37, 150, 3, (2, 3)), (36, 21, 21, (7,))]:
        fr = _frames(thr, variant, w, h)
        a, b = fr[0], fr[-1][::-1, ::-1]
        bo, wo = orc.match_wta(orc.edges(a, thr, variant), orc.edges(b, thr, variant), 1, sw, variant)
        for n in counts:
            _bands_check(orc, w, h, sw, n, a, b, thr, variant, bo, wo)
            with smb.MultiGpuBands(_devices(n), w, h, 1, sw, variant) as mb:
                web, best = mb.run(a, b, thr, want_best=True)
                assert np.array_equal(best, bo) and np.array_equal(web, wo), (w, h, sw, n)
                web, best = mb.run(a, b, thr, want_best=True, web16=True)
                assert np.array_equal(best, bo.astype(np.uint16)), (w, h, sw, n)


# ---- GHOST border rule ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("src", SOURCES)
@pytest.mark.parametrize("thr", THRS, ids=thr_id)
def test_ghost_border_rule(orc, thr, src):
    """A stencil that touches the ghost cells (128.0) always fires in frames of at least 2 x 2: the border ring is
    exactly 1 and a flat interior exactly 0, at every threshold."""
    for w, h in [(2, 2), (3, 2), (2, 3), (4, 4), (37, 5), (5, 37), (256, 9)]:
        with smb.StereoContext(w, h, 1, 1, smb.GHOST) as c:
            for v in (0, 100, 255):
                a = np.full((h, w), v, np.uint8)
                _load(c, a, a, src)
                c.edges(thr)
                e = c.download(smb.EDGES1)
                ring = np.ones((h, w), bool)
                ring[1:-1, 1:-1] = False
                assert (e[ring] == 1).all() and (e[~ring] == 0).all(), (w, h, v)
                assert np.array_equal(e, orc.edges(a, thr, smb.GHOST))


@pytest.mark.parametrize("thr", [1e-4, 2.5e-3], ids=thr_id)
def test_ghost_one_pixel_frames(orc, thr):
    """One-pixel-wide and one-pixel-high GHOST frames have ghost cells on both sides of a detector: the FP64 fallback
    of the gathering kernel decides on |a - b| of neighbouring pixels against the 128.0 cells.  Byte maps, and the
    planes alone through sm_run_batch."""
    rng = np.random.default_rng(17)
    for w, h in [(1, 200), (200, 1), (1, 1), (1, 5)]:
        imgs = np.stack([_small_frame(rng, w, h) for _ in range(18)])
        with smb.StereoContext(w, h, 1, 1, smb.GHOST) as c:
            for k in range(0, 18, 2):
                c.upload_u8(imgs[k], imgs[k + 1])
                _check_edges(orc, c, imgs[k], imgs[k + 1], thr, smb.GHOST, "u8")
            first, second = imgs[:17], np.concatenate([imgs[1:17], np.full((1, h, w), 128, np.uint8)])
            bo, wo = _want(orc, first, second, thr, smb.GHOST)
            c.set_option(smb.OPT_PIPE_GROUP, 3)
            web, best = c.run_batch(first, second, thr, want_best=True)
            assert np.array_equal(best, bo) and np.array_equal(web, wo), (w, h)


# ---- one context, the threshold switched between every kind of call ------------------------------------------------
@pytest.mark.parametrize("variant", [smb.WRAP, smb.GHOST], ids=vname)
def test_threshold_switching(orc, variant):
    """Every entry that detects edges rebuilds the context's table when the threshold changes, and they share one
    table: edges(t1), run_batch(t2), edges(t1), FP64 edges(t3), run_batch(t3), then band slots at t2 and t1."""
    w, h = 256, 120
    t1, t2, t3 = 1.0, 0.05, 0.4

    def edges(c, thr, src="u8"):
        fr = _frames(thr, variant, w, h)
        _load(c, fr[0], fr[-1], src)
        _check_edges(orc, c, fr[0], fr[-1], thr, variant, src)

    def batch(c, thr):
        first, second = _plane_pairs(thr, variant, w, h)
        bo, wo = _want(orc, first, second, thr, variant)
        web, best = c.run_batch(first, second, thr, want_best=True)
        assert np.array_equal(best, bo) and np.array_equal(web, wo), thr
        assert c.get_info(smb.INFO_EDGE_THRESHOLDS) == 1

    with smb.StereoContext(w, h, 1, 1, variant) as c:
        c.set_option(smb.OPT_PIPE_GROUP, 2)
        edges(c, t1)
        batch(c, t2)
        edges(c, t1)
        edges(c, t3, "fp64")
        c.set_option(smb.OPT_EDGES_FP64, 0)
        batch(c, t3)
    fr2, fr1 = _frames(t2, variant, w, h), _frames(t1, variant, w, h)
    with smb.MultiGpuBands(_devices(3), w, h, 1, 3, variant) as mb:
        for thr, fr in ((t2, fr2), (t1, fr1)):
            bo, wo = orc.match_wta(orc.edges(fr[0], thr, variant), orc.edges(fr[-1], thr, variant), 1, 3, variant)
            web, best = mb.run(fr[0], fr[-1], thr, want_best=True)
            assert np.array_equal(best, bo) and np.array_equal(web, wo), thr
