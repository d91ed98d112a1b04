"""The runner-up and web_sub from one launch of the hot kernel (k_bitslice_ru_sub, the *_ru_sub16 entries), on the GPU.

Every output of the combined entries -- best, web, runner_up and web_sub -- is compared bit for bit with
tests/extras_model.py and, where the test runs them on the same context, with the *_ru16 and *_sub16 entries'.  The
device entry writes between guard elements of 0xFFFF that must survive.  Covered: every reachable bit-sliced shape
family with m == 0 and m > 0 (the launched shape asserted equal to the 16-bit launch's), the 64-shift chunk boundaries,
the top of the sub-pixel range, the direct kernel's twin, row runs of many blocks forced through SM_OPT_ROW_RUNS, the
host-buffer entries (batch, multi-GPU batch, bands) and one context that switches among all six result formats."""
import numpy as np
import pytest

import stereomatching_b200 as smb
from extras_model import reference_all
from test_gpu_flavours import FLAVOURS, assert_shape, code, diff, expected_shape, run_dev_batch
from test_gpu_long_runs import assert_runs, cases
from test_gpu_min_shift import image_pair
from test_gpu_range_extras import F_D, F_H, F_M, F_SW, F_W, dev, inputs
from test_gpu_web16 import run16
from util import THRESHOLD, vname

pytestmark = pytest.mark.gpu

VARIANTS = [smb.WRAP, smb.GHOST]
GUARD = 41  # elements between one pair's frames and the next one's


@pytest.fixture(scope="module")
def num_sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def run_rs(c, les, res, with_best=True, rows=None):
    """sm_match_wta_dev_batch_ru_sub16 over distinct pairs, outputs out_stride = H*W + GUARD apart in buffers filled
    with 0xFFFF.  Asserts that nothing outside the frames (and, for a band context, outside its rows [r0, r1)) was
    written; returns (best or None, web, runner_up, web_sub) as (n, H, W) int32 arrays."""
    import torch
    n, (H, W) = len(les), les[0].shape
    npix, stride = H * W, H * W + GUARD
    d1 = torch.from_numpy(np.stack(les)).cuda()
    d2 = torch.from_numpy(np.stack(res)).cuda()
    fill = lambda: torch.full((n * stride + GUARD,), -1, dtype=torch.int16, device="cuda")  # noqa: E731  0xFFFF
    best, web, ru, ws = fill() if with_best else None, fill(), fill(), fill()
    torch.cuda.synchronize()
    c.match_wta_dev_batch_ru_sub16(n, d1.data_ptr(), d2.data_ptr(), npix, best.data_ptr() if with_best else None,
                                   web.data_ptr(), ru.data_ptr(), ws.data_ptr(), stride)
    c.synchronize()
    out = []
    for buf in (best, web, ru, ws):
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


def check(got, refs, what, ru=None, sub=None, rows=None):
    """got = (best or None, web, runner_up, web_sub) of n pairs against their reference_all tuples; ru / sub = the
    *_ru16 / *_sub16 entries' (best or None, web, extra) on the same inputs and context; rows = (r0, r1) compares
    those rows only."""
    r0, r1 = rows if rows is not None else (0, got[1].shape[1])
    for k, ref in enumerate(refs):
        w = "%s, pair %d" % (what, k)
        best, web, r, ws = (None if a is None else np.asarray(a[k][r0:r1], np.int32) for a in got)
        bo, wo, ro, so = (a[r0:r1] for a in ref)
        if best is not None:
            assert np.array_equal(best, bo), "%s: best %s" % (w, diff(best, bo))
        assert np.array_equal(web, wo), "%s: web %s" % (w, diff(web, wo))
        assert np.array_equal(r, ro), "%s: runner_up %s" % (w, diff(r, ro))
        assert np.array_equal(ws, so), "%s: web_sub %s" % (w, diff(ws, so))
        assert (r <= bo).all(), w + ": runner_up > best"
        assert np.array_equal((ws + 8) >> 4, web), w + ": web_sub does not round to web"
        for name, sib, mine in (("ru16", ru, r), ("sub16", sub, ws)):
            if sib is None:
                continue
            sb, sw_, sx = (None if a is None else np.asarray(a[k][r0:r1], np.int32) for a in sib)
            if best is not None and sb is not None:
                assert np.array_equal(best, sb), "%s: best != the %s entry's" % (w, name)
            assert np.array_equal(web, sw_), "%s: web != the %s entry's" % (w, name)
            assert np.array_equal(mine, sx), "%s: %s output differs" % (w, name)


# ---------------------------------------------------------------------------------
# A. every shape family, m == 0 and m > 0: one pair, several pairs, with and without best, a band
# ---------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
@pytest.mark.parametrize("flavour", list(FLAVOURS))
def test_shape_family(orc, num_sms, flavour, variant):
    nw, seg, multi, c2, hp, halves, geometry = FLAVOURS[flavour]
    for half in (halves[0], halves[len(halves) // 2]):
        W, H1, Hn, D = geometry(half, num_sms)
        sw = 2 * half + 1
        want = code(half, nw, seg, c2, hp, multi)
        one_pair = H1 <= 64
        H = H1 if one_pair else Hn
        for m in (0, 33, W + 5):
            tag = "%s half %d %dx%d D %d m %d %s" % (flavour, half, W, H, D, m, vname(variant))
            ins = inputs(W, H, D, m, 29 * m + W + D + half)
            refs = [reference_all(orc, name, le, re, D, sw, variant, m) for name, le, re in ins]
            if one_pair:
                with smb.StereoContext(W, H, D, sw, variant, kernel=smb.KERNEL_BITSLICE, min_shift=m) as c:
                    for k, (name, le, re) in enumerate(ins):
                        run16(c, [le], [re])
                        assert_shape(c, want, "%s %s 16-bit" % (tag, name))
                        sib_ru, sib_sub = dev(c, "ru", [le], [re]), dev(c, "sub", [le], [re])
                        for with_best in (True, False) if k < 2 else (True,):
                            what = "%s %s one pair%s" % (tag, name, "" if with_best else ", no best")
                            got = run_rs(c, [le], [re], with_best)
                            assert_shape(c, want, what)
                            check(got, refs[k:k + 1], what, sib_ru, sib_sub)
            if Hn is not None:
                with smb.StereoContext(W, Hn, D, sw, variant, kernel=smb.KERNEL_BITSLICE, min_shift=m) as c:
                    les, res = [f[1] for f in ins], [f[2] for f in ins]
                    run16(c, les, res)
                    assert_shape(c, want, tag + " 16-bit batch")
                    sib_ru, sib_sub = dev(c, "ru", les, res), dev(c, "sub", les, res)
                    for with_best in (True, False):
                        what = "%s, %d pairs per call%s" % (tag, len(ins), "" if with_best else ", no best")
                        got = run_rs(c, les, res, with_best)
                        assert c.get_info(smb.INFO_PAIRS_PER_LAUNCH) >= len(ins), what + ": not one launch"
                        assert_shape(c, want, what)
                        check(got, refs, what, sib_ru, sib_sub)
            # a band context: rows [r0, r1) only, the others keep their guard value
            r0, r1 = H // 3, H // 3 + max(1, min(H // 3, 20))
            band = expected_shape(W, r1 - r0, D, half, 1, num_sms)
            name, le, re = ins[1]
            with smb.StereoContext(W, H, D, sw, variant, rows=(r0, r1), kernel=smb.KERNEL_BITSLICE, min_shift=m) as c:
                what = "%s %s band [%d, %d)" % (tag, name, r0, r1)
                sib_ru = dev(c, "ru", [le], [re], True, rows=(r0, r1))
                got = run_rs(c, [le], [re], True, rows=(r0, r1))
                assert_shape(c, band, what)
                check(got, refs[1:2], what, sib_ru, rows=(r0, r1))


# ---------------------------------------------------------------------------------
# B. more than 64 shifts: winners on both sides of every chunk boundary and at both range ends
# ---------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
@pytest.mark.parametrize("D", [65, 129, 256])
def test_chunk_boundaries(orc, variant, D):
    W, H, sw = 384, 24, 9
    want = code(sw // 2, 2, 16, multi=True)
    for m in (0, 37):
        rng = np.random.default_rng(2000 * D + 10 * m + variant)
        ts = sorted({t for t in (0, 1, 62, 63, 64, 65, 127, 128, D - 2, D - 1) if t < D})
        ins = []
        for t in ts:
            le = (rng.random((H, W)) < 0.5).astype(np.uint8)
            ins.append(("winners on %d" % t, le, np.roll(le, m + t, axis=1) ^ (rng.random((H, W)) < 0.03).astype(np.uint8)))
        for P in (16, 64):
            le = np.tile((rng.random((H, P)) < 0.5).astype(np.uint8), (1, W // P))
            ins.append(("periodic%d" % P, le, le.copy()))
        refs = [reference_all(orc, "random", le, re, D, sw, variant, m) for _, le, re in ins]
        les, res = [f[1] for f in ins], [f[2] for f in ins]
        tag = "D %d m %d %s" % (D, m, vname(variant))
        with smb.StereoContext(W, H, D, sw, variant, min_shift=m) as c:
            for k, (name, le, re) in enumerate(ins):
                what = "%s %s one pair" % (tag, name)
                sib_ru, sib_sub = dev(c, "ru", [le], [re]), dev(c, "sub", [le], [re])
                got = run_rs(c, [le], [re])
                assert_shape(c, want, what)
                check(got, refs[k:k + 1], what, sib_ru, sib_sub)
            sib_ru, sib_sub = dev(c, "ru", les, res), dev(c, "sub", les, res)
            for with_best in (True, False):
                what = "%s batch%s" % (tag, "" if with_best else ", no best")
                got = run_rs(c, les, res, with_best)
                assert_shape(c, want, what)
                check(got, refs, what, sib_ru, sib_sub)
        # the inputs do what the test is about: most pixels win on the shift they were rolled by
        for k, t in enumerate(ts):
            on = refs[k][1] == m + t + 1
            assert on.mean() > (0.5 if variant == smb.WRAP else 0.2), (tag, t)


# ---------------------------------------------------------------------------------
# C. the top of the sub-pixel range
# ---------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
@pytest.mark.parametrize("kernel", [smb.KERNEL_AUTO, smb.KERNEL_DIRECT], ids=["auto", "direct"])
def test_top_of_the_range(orc, variant, kernel):
    """m + D == 4095 is accepted; m + D == 4096 is SM_ERR_ARG before any device call, from every entry."""
    W, H, sw = 64, 24, 9
    for D in (1, 65, 129):
        m = 4095 - D
        tag = "D %d m %d %s" % (D, m, vname(variant))
        ins = inputs(W, H, D, m, 4095 + D + variant)[:3]
        refs = [reference_all(orc, name, le, re, D, sw, variant, m) for name, le, re in ins]
        les, res = [f[1] for f in ins], [f[2] for f in ins]
        with smb.StereoContext(W, H, D, sw, variant, kernel=kernel, min_shift=m) as c:
            sib_ru, sib_sub = dev(c, "ru", les, res), dev(c, "sub", les, res)
            for with_best in (True, False):
                check(run_rs(c, les, res, with_best), refs, "%s, best %s" % (tag, with_best), sib_ru, sib_sub)
    D, m = 65, 4096 - 65
    z = np.zeros((1, H, W), np.uint8)
    with smb.StereoContext(W, H, D, sw, variant, kernel=kernel, min_shift=m) as c:
        buf = np.zeros(H * W, np.uint16)
        p = buf.ctypes.data
        rc = smb.lib().sm_match_wta_dev_batch_ru_sub16(c._c, 1, p, p, H * W, None, p, p, p, H * W)
        assert rc == -1 and b"4095" in smb.lib().sm_last_error()  # SM_ERR_ARG
        with pytest.raises(smb.StereoError):
            c.run_batch_ru_sub16(z, z)
        assert c.last_launches() == 0
    with smb.MultiGpuBatch([0], W, H, D, sw, variant, min_shift=m) as mb:
        with pytest.raises(smb.StereoError):
            mb.run_batch_ru_sub16(z, z)
    with smb.MultiGpuBands([0], W, H, D, sw, variant, min_shift=m) as bands:
        with pytest.raises(smb.StereoError):
            bands.run_ru_sub16(z[0], z[0])


# ---------------------------------------------------------------------------------
# D. the direct kernel's twin: forced, and the windows the auto kernel sends there
# ---------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
@pytest.mark.parametrize("W,H,D,sw,kernel", [(64, 40, 50, 9, smb.KERNEL_DIRECT), (64, 40, 130, 9, smb.KERNEL_DIRECT),
                                             (70, 66, 20, 33, smb.KERNEL_AUTO), (70, 66, 20, 47, smb.KERNEL_AUTO),
                                             (70, 66, 20, 63, smb.KERNEL_AUTO)],
                         ids=["forced_D50", "forced_D130", "window33", "window47", "window63"])
def test_direct_twin(orc, variant, W, H, D, sw, kernel):
    for m in (0, W + 3):
        tag = "%dx%d D %d window %d m %d %s" % (W, H, D, sw, m, vname(variant))
        ins = inputs(W, H, D, m, 19 * m + sw + D)[:3]
        refs = [reference_all(orc, name, le, re, D, sw, variant, m) for name, le, re in ins]
        les, res = [f[1] for f in ins], [f[2] for f in ins]
        with smb.StereoContext(W, H, D, sw, variant, kernel=kernel, min_shift=m) as c:
            sib_ru, sib_sub = dev(c, "ru", les, res), dev(c, "sub", les, res)
            got = run_rs(c, les[:1], res[:1])
            assert_shape(c, smb.SHAPE_DIRECT, tag + " one pair")
            check(got, refs[:1], tag + " one pair")
            for with_best in (True, False):
                got = run_rs(c, les, res, with_best)
                assert_shape(c, smb.SHAPE_DIRECT, tag)
                check(got, refs, "%s, best %s" % (tag, with_best), sib_ru, sib_sub)


# ---------------------------------------------------------------------------------
# E. row runs of many blocks: 7 whole blocks and a ragged one, the runs forced
# ---------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
@pytest.mark.parametrize("flavour", list(FLAVOURS))
def test_long_runs(orc, num_sms, flavour, variant):
    """One pair per launch with 1, 2, 3 and one run per block, then (16-pixel segments) all pairs in one launch with
    1 and 3 runs: the per-block prefetch of best, runner_up, web_sub and the carry past 64 shifts."""
    for half, W, H, D, m, RB, shape, ins in cases(orc, flavour, variant, num_sms):
        sw = 2 * half + 1
        max_runs = -(-H // RB)
        with smb.StereoContext(W, H, D, sw, variant, kernel=smb.KERNEL_BITSLICE, min_shift=m) as c:
            for name, le, re, ref in ins[:2]:
                for runs in (1, 2, 3, max_runs):
                    c.set_option(smb.OPT_ROW_RUNS, runs)
                    what = "%s half %d %dx%d D %d m %d %s %s, %d row runs asked" % (
                        flavour, half, W, H, D, m, vname(variant), name, runs)
                    got = run_rs(c, [le], [re], runs == 1)
                    assert_runs(c, shape, H, RB, runs, what)
                    check(got, [ref], what)
            if FLAVOURS[flavour][1] == 16:
                les, res, refs = [i[1] for i in ins], [i[2] for i in ins], [i[3] for i in ins]
                for runs in (1, 3):
                    c.set_option(smb.OPT_ROW_RUNS, runs)
                    what = "%s half %d %dx%d D %d m %d %s, %d pairs, %d row runs asked" % (
                        flavour, half, W, H, D, m, vname(variant), len(ins), runs)
                    got = run_rs(c, les, res)
                    assert c.get_info(smb.INFO_PAIRS_PER_LAUNCH) >= len(ins), what
                    assert_runs(c, shape, H, RB, runs, what)
                    check(got, refs, what)


# ---------------------------------------------------------------------------------
# F. the host-buffer entries from 8-bit images: batch in ragged pipeline stages, multi-GPU batch, bands
# ---------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
@pytest.mark.parametrize("W,H", [(128, 36), (67, 29)])
def test_host_entries(orc, variant, W, H):
    sw, n = 9, 5
    ndev = smb.device_count()
    devices = list(range(ndev)) if ndev > 1 else [0, 0, 0]  # (5 pairs over 3 slots: ragged shards)
    for D, m in ((16, 0), (40, 3), (100, W + 5)):
        tag = "%dx%d D %d m %d %s" % (W, H, D, m, vname(variant))
        pairs = [image_pair(orc, 8765 + 2 * k + m + D, W, H, m, D) for k in range(n)]
        first = np.stack([p[0] for p in pairs])
        second = np.stack([p[1] for p in pairs])
        refs = [reference_all(orc, "random", orc.edges(p[0], THRESHOLD, variant), orc.edges(p[1], THRESHOLD, variant),
                              D, sw, variant, m) for p in pairs]
        with smb.StereoContext(W, H, D, sw, variant, min_shift=m) as c:
            c.set_option(smb.OPT_PIPE_GROUP, 2)  # several stages, a ragged last one
            web, best, ru = c.run_batch(first, second, THRESHOLD, want_best=True, web16=True, want_runner_up=True)
            sib_ru = (best, web, ru)
            web, best, ws = c.run_batch(first, second, THRESHOLD, want_best=True, web16=True, want_subpixel=True)
            sib_sub = (best, web, ws)
            web, best, ru, ws = c.run_batch_ru_sub16(first, second, THRESHOLD, want_best=True)
            assert all(a.dtype == np.uint16 for a in (web, best, ru, ws))
            check((best, web, ru, ws), refs, tag + " run_batch_ru_sub16", sib_ru, sib_sub)
            web, ru, ws = c.run_batch_ru_sub16(first, second, THRESHOLD)
            check((None, web, ru, ws), refs, tag + " run_batch_ru_sub16, no best", sib_ru, sib_sub)
        with smb.MultiGpuBatch(devices, W, H, D, sw, variant, min_shift=m) as mb:
            web, best, ru, ws = mb.run_batch_ru_sub16(first, second, THRESHOLD, want_best=True)
            check((best, web, ru, ws), refs, "%s multi %s" % (tag, devices), sib_ru, sib_sub)
            web, ru, ws = mb.run_batch_ru_sub16(first, second, THRESHOLD)
            check((None, web, ru, ws), refs, "%s multi %s, no best" % (tag, devices), sib_ru, sib_sub)
        for nb in (1, 2, 3):
            with smb.MultiGpuBands([0] * nb, W, H, D, sw, variant, min_shift=m) as bands:
                web, best, ru, ws = bands.run_ru_sub16(first[0], second[0], THRESHOLD, want_best=True)
                check((best[None], web[None], ru[None], ws[None]), refs[:1], "%s %d bands" % (tag, nb))
                web, ru, ws = bands.run_ru_sub16(first[0], second[0], THRESHOLD)
                check((None, web[None], ru[None], ws[None]), refs[:1], "%s %d bands, no best" % (tag, nb))


# ---------------------------------------------------------------------------------
# G. one context, all six result formats in sequence: the launch counts of a fresh context
# ---------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
def test_one_context_every_format(orc, variant):
    """int32, u8, u16, runner-up, sub-pixel and both, through the host entries; and the device entries.  At D 100,
    window 13 the MULTI extra families hold fewer CTAs per SM than the int32 / 16-bit ones, so their launches take
    fewer pairs, which shows in the launch counts."""
    n, few, distinct = 29, 7, 3
    pairs = [image_pair(orc, 900 + 2 * k + variant, F_W, F_H, F_M, F_D) for k in range(distinct)]
    edges = [(orc.edges(p[0], THRESHOLD, variant), orc.edges(p[1], THRESHOLD, variant)) for p in pairs]
    refs = [reference_all(orc, "random", e[0], e[1], F_D, F_SW, variant, F_M) for e in edges]
    refs = [refs[k % distinct] for k in range(n)]
    first = np.stack([pairs[k % distinct][0] for k in range(n)])
    second = np.stack([pairs[k % distinct][1] for k in range(n)])
    les = [edges[k % distinct][0] for k in range(n)]
    res = [edges[k % distinct][1] for k in range(n)]

    def i32(c):
        web, best = c.run_batch(first, second, THRESHOLD, want_best=True)
        for j in range(n):
            assert np.array_equal(best[j], refs[j][0]) and np.array_equal(web[j], refs[j][1]), ("i32", j)

    def u8(c):
        web = c.run_batch(first, second, THRESHOLD, web_u8=True)
        for j in range(n):
            assert np.array_equal(web[j], refs[j][1].astype(np.uint8)), ("u8", j)

    def u16(c):
        web = c.run_batch(first, second, THRESHOLD, web16=True)
        for j in range(n):
            assert np.array_equal(web[j].astype(np.int32), refs[j][1]), ("u16", j)

    def ru(c, k=n):
        web, best, r = c.run_batch(first[:k], second[:k], THRESHOLD, want_best=True, web16=True, want_runner_up=True)
        for j in range(k):
            assert np.array_equal(r[j].astype(np.int32), refs[j][2]) and np.array_equal(web[j], refs[j][1]), ("ru", j)

    def sub(c):
        web, ws = c.run_batch(first, second, THRESHOLD, web16=True, want_subpixel=True)
        for j in range(n):
            assert np.array_equal(ws[j].astype(np.int32), refs[j][3]) and np.array_equal(web[j], refs[j][1]), ("sub", j)

    def both(with_best, k=n):
        def call(c):
            out = c.run_batch_ru_sub16(first[:k], second[:k], THRESHOLD, want_best=with_best)
            got = (out[1], out[0], out[2], out[3]) if with_best else (None,) + tuple(out)
            check(got, refs[:k], "run_batch_ru_sub16 %d pairs" % k)
        return call

    def both_dev(c):
        check(run_rs(c, les, res), refs, "match_wta_dev_batch_ru_sub16")

    def i32_dev(c):
        best, web = run_dev_batch(c, les, res)
        for j in range(n):
            assert np.array_equal(best[j], refs[j][0]) and np.array_equal(web[j], refs[j][1]), ("i32 dev", j)

    steps = [("i32", i32), ("ru_sub16", both(True)), ("u16", u16), ("ru16", ru), ("ru_sub16 without best", both(False)),
             ("sub16", sub), ("u8", u8), ("ru_sub16 fewer pairs", both(True, few)), ("ru16 fewer pairs",
             lambda c: ru(c, few)), ("ru_sub16 device", both_dev), ("i32 device", i32_dev), ("i32 again", i32)]
    fresh = {}
    for name, step in steps:
        with smb.StereoContext(F_W, F_H, F_D, F_SW, variant, min_shift=F_M) as c:
            step(c)
            fresh[name] = c.last_launches()
    assert fresh["ru_sub16"] > fresh["i32"], fresh
    with smb.StereoContext(F_W, F_H, F_D, F_SW, variant, min_shift=F_M) as c:
        for name, step in steps:
            step(c)
            assert c.last_launches() == fresh[name], "%s after the others: %d launches, %d on a fresh context" % (
                name, c.last_launches(), fresh[name])
