"""The sub-pixel entries on the GPU: sm_match_wta_dev_batch_sub16 (the k_bitslice_sub / k_direct16_sub kernels),
sm_run_batch_sub16, sm_multi_run_batch_sub16 and sm_bands_run_sub16.

Every reachable instantiation of the sub-pixel family runs the flavour table of test_gpu_flavours.py in one-pair
and several-pairs launches, with and without best: web_sub equals the reference model's
(tests/subpixel_model.py, the contract's parabola vertex over the oracle's score planes), best / web equal the 16-bit entry's on
the same inputs, and the launch reports the 16-bit launch's shape.  Outputs sit in buffers whose pairs are further
apart than a frame, with guard elements of 0xFFFF that must survive every launch."""
import numpy as np
import pytest

import oracle
import stereomatching_b200 as smb
from subpixel_model import match_wta_sub, reference_sub
from test_gpu_flavours import FLAVOURS, REACHABLE, code, expected_shape, families
from util import THRESHOLD, vname

pytestmark = pytest.mark.gpu

VARIANTS = [smb.WRAP, smb.GHOST]
GUARD = 37      # elements between one pair's frame and the next one's
SEEN_SUB = set()  # shape codes of the sub-pixel launches compared with the model by test_flavour_sub
DONE_SUB = set()


@pytest.fixture(scope="module")
def num_sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def run_dev(c, les, res, with_best=True, rows=None, sub=True):
    """sm_match_wta_dev_batch_sub16 (sub: the sub-pixel entry) or sm_match_wta_dev_batch16 over distinct pairs, outputs out_stride = H*W +
    GUARD apart in buffers filled with 0xFFFF.  Asserts that nothing outside the frames (and, for a band context,
    outside its rows [r0, r1)) was written; returns (best, web, web_sub) as (n, H, W) int32 arrays (best None
    without, web_sub None for the 16-bit entry)."""
    import torch
    n, (H, W) = len(les), les[0].shape
    npix, stride = H * W, H * W + GUARD
    d1 = torch.from_numpy(np.stack(les)).cuda()
    d2 = torch.from_numpy(np.stack(res)).cuda()
    fill = lambda: torch.full((n * stride + GUARD,), -1, dtype=torch.int16, device="cuda")  # noqa: E731  0xFFFF
    web, best, wsub = fill(), fill() if with_best else None, fill() if sub else None
    torch.cuda.synchronize()
    bp = best.data_ptr() if with_best else None
    if sub:
        c.match_wta_dev_batch_sub16(n, d1.data_ptr(), d2.data_ptr(), npix, bp, web.data_ptr(), wsub.data_ptr(), stride)
    else:
        c.match_wta_dev_batch16(n, d1.data_ptr(), d2.data_ptr(), npix, bp, web.data_ptr(), stride)
    c.synchronize()
    out = []
    for buf in (best, web, wsub):
        if buf is None:
            out.append(None)
            continue
        a = buf.cpu().numpy().view(np.uint16)
        frames = np.stack([a[k * stride:k * stride + npix] for k in range(n)]).reshape(n, H, W)
        guards = np.concatenate([a[k * stride + npix:(k + 1) * stride] for k in range(n)] + [a[n * stride:]])
        assert (guards == 0xFFFF).all(), "%d guard elements written" % (guards != 0xFFFF).sum()
        if rows is not None:
            r0, r1 = rows
            outside = np.concatenate([frames[:, :r0].ravel(), frames[:, r1:].ravel()])
            assert (outside == 0xFFFF).all(), "a band context wrote outside its rows"
        out.append(frames.astype(np.int32))
    return tuple(out)


def diff(got, want):
    bad = np.argwhere(got != want)
    return "%d pixels differ, first (y, x) %s: %s != %s" % (
        len(bad), tuple(bad[0]), got[tuple(bad[0])], want[tuple(bad[0])]) if len(bad) else "equal"


def check(best, web, ws, ref, what):
    """best / web / web_sub against a reference (best, web, web_sub); best may be None."""
    bo, wo, so = ref
    if best is not None:
        assert np.array_equal(best, bo), "%s: best %s" % (what, diff(best, bo))
    assert np.array_equal(web, wo), "%s: web %s" % (what, diff(web, wo))
    assert np.array_equal(ws, so), "%s: web_sub %s" % (what, diff(ws, so))
    assert np.array_equal((ws + 8) >> 4, web), what


def at(a, k):
    return None if a is None else a[k]


# ---------------------------------------------------------------------------------
# every reachable k_bitslice_sub instantiation
# ---------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
@pytest.mark.parametrize("flavour", list(FLAVOURS))
def test_flavour_sub(orc, num_sms, flavour, variant):
    nw, seg, multi, c2, hp, halves, geometry = FLAVOURS[flavour]
    for half in halves:
        want = code(half, nw, seg, c2, hp, multi)
        W, H1, Hn, D = geometry(half, num_sms)
        sw = 2 * half + 1
        seed = 9000 + 1000 * half + 17 * D + W
        tag = "%s half %d %dx%d D %d %s" % (flavour, half, W, H1, D, vname(variant))
        fams = families(W, H1, D, seed)
        refs = {name: reference_sub(orc, name, le, re, D, sw, variant) for name, le, re in fams}
        with smb.StereoContext(W, H1, D, sw, variant, kernel=smb.KERNEL_BITSLICE) as c:
            # the 16-bit entry's one-pair launch on the first input: the sub-pixel one reports its shape
            b16, w16, _ = run_dev(c, [fams[0][1]], [fams[0][2]], sub=False)
            shape16 = c.get_info(smb.INFO_KERNEL_SHAPE)
            assert shape16 == want, tag
            for k, (name, le, re) in enumerate(fams):
                for with_best in (True, False) if k < 2 else (True,):
                    best, web, sub = run_dev(c, [le], [re], with_best)
                    what = "%s %s one pair%s" % (tag, name, "" if with_best else ", no best")
                    assert c.get_info(smb.INFO_KERNEL_SHAPE) == shape16, what
                    SEEN_SUB.add(c.get_info(smb.INFO_KERNEL_SHAPE))
                    check(at(best, 0), web[0], sub[0], refs[name], what)
                    if k == 0:
                        check(at(best, 0), web[0], sub[0], (b16[0], w16[0], refs[name][2]), what + " vs 16-bit")
        if Hn is not None:
            if Hn != H1:
                fams = families(W, Hn, D, seed + 1)
                refs = {name: reference_sub(orc, name, le, re, D, sw, variant) for name, le, re in fams}
            with smb.StereoContext(W, Hn, D, sw, variant, kernel=smb.KERNEL_BITSLICE) as c:
                les, res = [f[1] for f in fams], [f[2] for f in fams]
                b16, w16, _ = run_dev(c, les, res, sub=False)
                shape16 = c.get_info(smb.INFO_KERNEL_SHAPE)
                for with_best in (True, False):
                    best, web, sub = run_dev(c, les, res, with_best)
                    what = "%s, %d pairs per call%s" % (tag, len(fams), "" if with_best else ", no best")
                    assert c.get_info(smb.INFO_KERNEL_SHAPE) == shape16 == want, what
                    SEEN_SUB.add(want)
                    for k, (name, _, _) in enumerate(fams):
                        check(at(best, k), web[k], sub[k], refs[name], "%s, pair %d (%s)" % (what, k, name))
                        check(at(best, k), web[k], sub[k], (b16[k], w16[k], refs[name][2]), "%s, pair %d vs 16-bit"
                              % (what, k))
        # a band context: rows [r0, r1) only, the others keep their guard value
        name, le, re = fams[1] if Hn is None or Hn == H1 else families(W, H1, D, seed)[1]
        ref = reference_sub(orc, name, le, re, D, sw, variant)
        r0, r1 = H1 // 3, H1 // 3 + max(1, min(H1 // 3, 20))
        with smb.StereoContext(W, H1, D, sw, variant, rows=(r0, r1), kernel=smb.KERNEL_BITSLICE) as c:
            best, web, sub = run_dev(c, [le], [re], True, rows=(r0, r1))
            assert c.get_info(smb.INFO_KERNEL_SHAPE) == expected_shape(W, r1 - r0, D, half, 1, num_sms)
        check(best[0, r0:r1], web[0, r0:r1], sub[0, r0:r1], tuple(a[r0:r1] for a in ref),
              "%s band [%d, %d)" % (tag, r0, r1))
    DONE_SUB.add((flavour, variant))


# ---------------------------------------------------------------------------------
# more than 64 shifts: the chunks merge (best, web, web_sub) through the u16 arrays and the carry
# ---------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
@pytest.mark.parametrize("D", [65, 129, 256, 512])
def test_multi_chunks(orc, variant, D):
    """Maps periodic in x with periods 16, 32 and 64 tie across every 64-shift chunk boundary."""
    W, H, sw = 128, 24, 9
    fams = [f for f in families(W, H, D, 41 * D + variant) if f[0].startswith("periodic") or f[0] == "random0.60"]
    assert len(fams) == 4
    refs = {name: reference_sub(orc, name, le, re, D, sw, variant) for name, le, re in fams}
    with smb.StereoContext(W, H, D, sw, variant) as c:
        for with_best in (True, False):
            for name, le, re in fams:  # one pair per launch
                best, web, sub = run_dev(c, [le], [re], with_best)
                assert c.get_info(smb.INFO_KERNEL_SHAPE) & smb.SHAPE_MULTI
                check(at(best, 0), web[0], sub[0], refs[name], "D %d %s one pair, best %s" % (D, name, with_best))
            best, web, sub = run_dev(c, [f[1] for f in fams], [f[2] for f in fams], with_best)
            for k, (name, _, _) in enumerate(fams):
                check(at(best, k), web[k], sub[k], refs[name], "D %d %s in a batch, best %s" % (D, name, with_best))


@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
@pytest.mark.parametrize("W,H,D,sw", [(48, 40, 30, 21), (64, 40, 129, 9)], ids=["one_word", "chunks"])
def test_ragged_batch(orc, variant, W, H, D, sw):
    """17 pairs: a launch of 16, then one of a single pair, with and without best; best / web are the 16-bit
    entry's, web_sub the model's."""
    n = 17
    rng = np.random.default_rng(270 + D + variant)
    les = [(rng.random((H, W)) < (0.1 + 0.04 * k)).astype(np.uint8) for k in range(n)]
    res = [np.roll(le, k % D, axis=1) ^ (rng.random((H, W)) < 0.02).astype(np.uint8) for k, le in enumerate(les)]
    with smb.StereoContext(W, H, D, sw, variant) as c:
        b16, w16, _ = run_dev(c, les, res, sub=False)
        shape16, runs16 = c.get_info(smb.INFO_KERNEL_SHAPE), c.get_info(smb.INFO_ROW_RUNS)
        assert c.get_info(smb.INFO_PAIRS_PER_LAUNCH) == 16
        # the 16-bit batch ends on a one-pair launch: alone it takes the latency mode's shape and row runs
        run_dev(c, les[16:], res[16:], sub=False)
        assert (c.get_info(smb.INFO_KERNEL_SHAPE), c.get_info(smb.INFO_ROW_RUNS)) == (shape16, runs16)
        for with_best in (True, False):
            best, web, sub = run_dev(c, les, res, with_best)
            # 16 + 1: two groups (a pack and a main kernel each), the last a one-pair launch like the 16-bit one's
            assert (c.get_info(smb.INFO_KERNEL_SHAPE), c.get_info(smb.INFO_ROW_RUNS)) == (shape16, runs16)
            assert c.last_launches() == 4
            run_dev(c, les[:16], res[:16], with_best)
            assert c.last_launches() == 2, "the sub-pixel batch of 16 pairs is not one launch"
            for k in range(n):
                if with_best:
                    assert np.array_equal(best[k], b16[k]), k
                assert np.array_equal(web[k], w16[k]), k
            for k in (0, 15, 16):
                check(at(best, k), web[k], sub[k], reference_sub(orc, "random", les[k], res[k], D, sw, variant),
                      "pair %d, best %s" % (k, with_best))


# ---------------------------------------------------------------------------------
# the direct kernel's twin, min_shift, one shift, saturated maps
# ---------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
@pytest.mark.parametrize("sw", [33, 45, 63])
def test_direct_wide_windows(orc, variant, sw):
    W, H, D = 70, 66, 20
    name, le, re = families(W, H, D, sw + variant)[1]
    ref = reference_sub(orc, name, le, re, D, sw, variant)
    with smb.StereoContext(W, H, D, sw, variant) as c:
        for with_best in (True, False):
            best, web, sub = run_dev(c, [le, le], [re, re], with_best)
            assert c.get_info(smb.INFO_KERNEL_SHAPE) == smb.SHAPE_DIRECT
            for k in range(2):
                check(at(best, k), web[k], sub[k], ref, "window %d, best %s" % (sw, with_best))


@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
def test_direct_forced(orc, variant):
    W, H, D, sw = 64, 40, 50, 9
    fams = families(W, H, D, 60 + variant)
    with smb.StereoContext(W, H, D, sw, variant, kernel=smb.KERNEL_DIRECT) as c:
        les, res = [f[1] for f in fams], [f[2] for f in fams]
        for with_best in (True, False):
            best, web, sub = run_dev(c, les, res, with_best)
            assert c.get_info(smb.INFO_KERNEL_SHAPE) == smb.SHAPE_DIRECT
            for k, (name, le, re) in enumerate(fams):
                check(at(best, k), web[k], sub[k], reference_sub(orc, name, le, re, D, sw, variant), name)


@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
@pytest.mark.parametrize("W,H,D,sw,m", [(64, 40, 50, 9, 7), (160, 40, 13, 5, 33), (48, 40, 30, 21, 3)],
                         ids=["two_words", "column_half_word_pairs", "one_word"])
def test_min_shift(orc, num_sms, variant, W, H, D, sw, m):
    """A search range [m, m + D): the model runs over the oracle's score planes of shifts m .. m + D - 1 (the second
    map offset by the planes' producers, as test_gpu_min_shift.py checks it)."""
    rng = np.random.default_rng(W + m + variant)
    les = [(rng.random((H, W)) < d).astype(np.uint8) for d in (0.2, 0.6)]
    res = [np.roll(le, m + k + 2, axis=1) ^ (rng.random((H, W)) < 0.05).astype(np.uint8) for k, le in enumerate(les)]
    refs = [match_wta_sub(orc, le, re, D, sw, variant, m=m) for le, re in zip(les, res)]
    with smb.StereoContext(W, H, D, sw, variant, min_shift=m) as c:
        for n in (1, 2):
            best, web, sub = run_dev(c, les[:n], res[:n])
            for k in range(n):
                check(best[k], web[k], sub[k], refs[k], "min_shift %d, %d pairs, pair %d" % (m, n, k))


@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
@pytest.mark.parametrize("W,sw", [(48, 9), (128, 5), (160, 3), (70, 33)])
def test_one_shift_has_no_fraction(orc, variant, W, sw):
    H = 40
    rng = np.random.default_rng(W + sw)
    le = (rng.random((H, W)) < 0.5).astype(np.uint8)
    with smb.StereoContext(W, H, 1, sw, variant) as c:
        best, web, sub = run_dev(c, [le, le], [le, np.roll(le, 1, axis=1)])
    assert np.array_equal(sub, 16 * web)
    assert (web == 1).all()


@pytest.mark.parametrize("W,D,sw", [(48, 30, 21), (64, 50, 9), (64, 130, 7), (128, 30, 9), (160, 16, 5), (100, 16, 29),
                                    (70, 20, 33)])
def test_saturated_wrap_sits_on_the_last_shift(W, D, sw):
    H = 40
    z = np.zeros((H, W), np.uint8)
    with smb.StereoContext(W, H, D, sw, smb.WRAP) as c:
        best, web, sub = run_dev(c, [z, z], [z, z])
    assert (best == sw * sw).all() and (sub == 16 * D).all() and (web == D).all()


@pytest.mark.parametrize("W,D,sw", [(64, 50, 9), (128, 30, 9), (64, 130, 7)])
def test_saturated_ghost_borders(orc, W, D, sw):
    H = 40
    z = np.zeros((H, W), np.uint8)
    with smb.StereoContext(W, H, D, sw, smb.GHOST) as c:
        best, web, sub = run_dev(c, [z], [z])
    check(best[0], web[0], sub[0], reference_sub(orc, "saturated", z, z, D, sw, smb.GHOST), "ghost saturated")


@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
@pytest.mark.parametrize("D", [65, 129, 256, 512])
def test_multi_chunk_boundaries(orc, variant, D):
    """Right maps rolled so that winners sit on shifts 63, 64, 127, 128 and D - 1: on both sides of every chunk
    boundary and at the range's end; a large share of those pixels has a non-zero fraction."""
    W, H, sw = 704, 24, 9  # wider than every shift: a roll has one best shift, also in WRAP
    rng = np.random.default_rng(77 * D + variant)
    shifts = sorted({s for s in (63, 64, 127, 128, D - 1) if s < D})
    les = [(rng.random((H, W)) < 0.5).astype(np.uint8) for _ in shifts]
    # a few flipped pixels keep the neighbours' scores apart, so that fractions are non-zero
    res = [np.roll(le, s, axis=1) ^ (rng.random((H, W)) < 0.03).astype(np.uint8) for le, s in zip(les, shifts)]
    refs = [reference_sub(orc, "random", le, re, D, sw, variant) for le, re in zip(les, res)]
    with smb.StereoContext(W, H, D, sw, variant) as c:
        for with_best in (True, False):
            for k, s in enumerate(shifts):
                best, web, ws = run_dev(c, [les[k]], [res[k]], with_best)
                assert c.get_info(smb.INFO_KERNEL_SHAPE) & smb.SHAPE_MULTI
                check(at(best, 0), web[0], ws[0], refs[k], "D %d winners on %d, one pair" % (D, s))
            best, web, ws = run_dev(c, les, res, with_best)
            for k, s in enumerate(shifts):
                check(at(best, k), web[k], ws[k], refs[k], "D %d winners on %d, batch" % (D, s))
    for k, s in enumerate(shifts):
        on = refs[k][1] == s + 1
        assert on.mean() > 0.2, (D, s)  # (GHOST: a roll by s leaves s columns without a match)
        if s != D - 1:
            assert (refs[k][2][on] % 16 != 0).mean() > 0.3, (D, s)  # the test cannot pass on zeros
        else:
            assert (refs[k][2][on] == 16 * D).all()


@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
@pytest.mark.parametrize("W,D,sw", [(48, 30, 21), (128, 30, 9), (160, 16, 5)], ids=["one_word", "column_pairs",
                                                                                     "half_word_pairs"])
def test_range_ends(orc, num_sms, variant, W, D, sw):
    """Winners on the first and on the last shift, with non-zero inner neighbours: frac == 0 there."""
    H = 40
    rng = np.random.default_rng(W + D + variant)
    les = [(rng.random((H, W)) < 0.5).astype(np.uint8) for _ in range(2)]
    res = [np.roll(les[0], 0, axis=1), np.roll(les[1], D - 1, axis=1)]
    refs = [reference_sub(orc, "random", le, re, D, sw, variant) for le, re in zip(les, res)]
    with smb.StereoContext(W, H, D, sw, variant) as c:
        best, web, ws = run_dev(c, les, res)
        b16, w16, _ = run_dev(c, les, res, sub=False)
        assert c.get_info(smb.INFO_KERNEL_SHAPE) == expected_shape(W, H, D, sw // 2, 2, num_sms)
    for k, end in enumerate((1, D)):
        check(best[k], web[k], ws[k], refs[k], "winner on shift %d" % (end - 1))
        assert np.array_equal(best[k], b16[k]) and np.array_equal(web[k], w16[k])
        on = web[k] == end
        assert on.mean() > 0.5
        assert (ws[k][on] == 16 * end).all()


@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
def test_range_limit(variant):
    """m + D == 4095 is accepted, 4096 rejected with SM_ERR_ARG before the device (web_sub fits 16 bits)."""
    import torch
    W, H, D, sw = 64, 24, 40, 9
    rng = np.random.default_rng(4095 + variant)
    le = (rng.random((H, W)) < 0.5).astype(np.uint8)
    re = np.roll(le, 5, axis=1)
    with smb.StereoContext(W, H, D, sw, variant, min_shift=4095 - D) as c:
        best, web, ws = run_dev(c, [le], [re])
        assert (web >= 4095 - D + 1).all() and (web <= 4095).all()
        assert np.array_equal((ws + 8) >> 4, web) and (ws <= 0xFFFF).all()
    with smb.StereoContext(W, H, D, sw, variant, min_shift=4096 - D) as c:
        e = torch.zeros((H, W), dtype=torch.uint8, device="cuda")
        o = torch.zeros((H * W,), dtype=torch.int16, device="cuda")
        with pytest.raises(smb.StereoError, match="4095"):
            c.match_wta_dev_batch_sub16(1, e.data_ptr(), e.data_ptr(), H * W, None, o.data_ptr(), o.data_ptr(), H * W)
        z = np.zeros((1, H, W), np.uint8)
        with pytest.raises(smb.StereoError, match="4095"):
            c.run_batch(z, z, web16=True, want_subpixel=True)
    with smb.MultiGpuBatch([0], W, H, D, sw, variant, min_shift=4096 - D) as m:
        with pytest.raises(smb.StereoError, match="4095"):
            m.run_batch(z, z, web16=True, want_subpixel=True)
    with smb.MultiGpuBands([0, 0], W, H, D, sw, variant, min_shift=4096 - D) as b:
        with pytest.raises(smb.StereoError, match="4095"):
            b.run(z[0], z[0], web16=True, want_subpixel=True)


# ---------------------------------------------------------------------------------
# host-buffer entries
# ---------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
def test_config4_batch_sub16(orc, golden, variant):
    """Config 4 (1280x720, 128 shifts, window 21): the four reference-pinned pairs repeated to 10 through
    sm_run_batch_sub16 and sm_multi_run_batch_sub16 (slots [0, 0]); web / best against the reference's CRCs, web_sub
    against the model on the oracle's edge maps."""
    gs = [golden["synth/c4/%d/%s" % (k, vname(variant))] for k in range(4)]
    pairs = [orc.synth_pair(g["seed"], g["w"], g["h"], g["D"]) for g in gs]
    n = 10
    first = np.stack([pairs[k % 4][0] for k in range(n)])
    second = np.stack([pairs[k % 4][1] for k in range(n)])
    g0 = gs[0]
    with smb.StereoContext(g0["w"], g0["h"], g0["D"], g0["sw"], variant) as c:
        web, best, sub = c.run_batch(first, second, THRESHOLD, want_best=True, web16=True, want_subpixel=True)
        web_only, ws_only = c.run_batch(first, second, THRESHOLD, web16=True, want_subpixel=True)
        web16 = c.run_batch(first, second, THRESHOLD, web16=True)
    with smb.MultiGpuBatch([0, 0], g0["w"], g0["h"], g0["D"], g0["sw"], variant) as m:
        mweb, mbest, mws = m.run_batch(first, second, THRESHOLD, want_best=True, web16=True, want_subpixel=True)
    for k in range(n):
        for w_, b_, r_ in ((web, best, sub), (mweb, mbest, mws)):
            assert w_.dtype == b_.dtype == r_.dtype == np.uint16
            assert oracle.crc32(w_[k].astype(np.int32)) == gs[k % 4]["web"], k
            assert oracle.crc32(b_[k].astype(np.int32)) == gs[k % 4]["best"], k
            assert np.array_equal((r_[k].astype(np.int32) + 8) >> 4, w_[k].astype(np.int32)), k
    assert np.array_equal(web_only, web) and np.array_equal(ws_only, sub) and np.array_equal(web16, web)
    assert np.array_equal(mws, sub)
    for k in range(4):
        e1 = orc.edges(pairs[k][0], THRESHOLD, variant)
        e2 = orc.edges(pairs[k][1], THRESHOLD, variant)
        bo, wo, ro = match_wta_sub(orc, e1, e2, g0["D"], g0["sw"], variant)
        assert np.array_equal(best[k].astype(np.int32), bo), k
        assert np.array_equal(sub[k].astype(np.int32), ro), "pair %d: web_sub %s" % (k, diff(sub[k].astype(np.int32), ro))


@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
def test_config3_bands_sub16(orc, golden, variant):
    """Config 3 (3840x2160, 256 shifts, window 11) through sm_bands_run_sub16, every slot on device 0: 1, 2 and 8
    bands; web_sub is the same whatever the bands."""
    g = golden["synth/c3/%s" % vname(variant)]
    left, right, _ = orc.synth_pair(g["seed"], g["w"], g["h"], g["D"])
    wss = []
    for nb in (1, 2, 8):
        with smb.MultiGpuBands([0] * nb, g["w"], g["h"], g["D"], g["sw"], variant) as b:
            web, best, sub = b.run(left, right, THRESHOLD, want_best=True, web16=True, want_subpixel=True)
            assert web.dtype == best.dtype == sub.dtype == np.uint16
            assert oracle.crc32(web.astype(np.int32)) == g["web"], nb
            assert oracle.crc32(best.astype(np.int32)) == g["best"], nb
            assert np.array_equal((sub.astype(np.int32) + 8) >> 4, web.astype(np.int32)), nb
            web_only, ws_only = b.run(left, right, THRESHOLD, web16=True, want_subpixel=True)
            assert np.array_equal(web_only, web) and np.array_equal(ws_only, sub), nb
            wss.append(sub)
    assert np.array_equal(wss[0], wss[1]) and np.array_equal(wss[0], wss[2])


def test_arguments_with_a_context():
    import torch
    W, H = 64, 32
    L = smb.lib()
    e = torch.zeros((2, H, W), dtype=torch.uint8, device="cuda")
    o = torch.zeros((2, H * W), dtype=torch.int16, device="cuda")
    with smb.StereoContext(W, H, 40, 9) as c:
        with pytest.raises(smb.StereoError, match="stride below frame size"):
            c.match_wta_dev_batch_sub16(1, e.data_ptr(), e.data_ptr(), H * W, None, o.data_ptr(), o.data_ptr(), H * W - 1)
        c.match_wta_dev_batch_sub16(0, e.data_ptr(), e.data_ptr(), H * W, None, o.data_ptr(), o.data_ptr(), H * W)
    with smb.StereoContext(W, H, 40, 9, rows=(4, 20)) as c:
        z = np.zeros((1, H, W), np.uint8)
        with pytest.raises(smb.StereoError, match="whole-frame contexts only"):
            c.run_batch(z, z, web16=True, want_subpixel=True)
        r = np.zeros((1, H, W), np.uint16)
        assert L.sm_run_batch_sub16(c._c, 1, z.ctypes.data, z.ctypes.data, 0.15, r.ctypes.data, None, None) == -1


def test_every_reachable_kernel_ran_with_web_sub():
    """Runs last: test_flavour_sub launched exactly the reachable set of k_bitslice_sub instantiations."""
    if len(DONE_SUB) < len(FLAVOURS) * len(VARIANTS):
        pytest.skip("needs every test_flavour_sub case of this session to have passed")
    assert SEEN_SUB == REACHABLE, "missing %s, unexpected %s" % (
        sorted(hex(x) for x in REACHABLE - SEEN_SUB), sorted(hex(x) for x in SEEN_SUB - REACHABLE))
