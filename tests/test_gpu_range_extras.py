"""The runner-up and sub-pixel results over search ranges that start above zero, on the GPU.

Each of the hot path's result families (int32, 16-bit, runner-up, sub-pixel) was tested hard on its own, mostly with
the others at their defaults.  Here they meet: a range [m, m + D) with m > 0 through every bit-sliced shape family
(asserted through SM_INFO_KERNEL_SHAPE, the MULTI chunk merge included), the chunk boundaries of ranges of more than 64
shifts, the direct kernel's twins, the top of each family's range, the host-buffer entries from 8-bit images (batch,
multi-GPU batch, bands), one context that switches between every family, and a seeded random sample.

Every runner-up and sub-pixel result is compared bit for bit with tests/extras_model.py (all four outputs from one
stack of the oracle's score planes), and its best / web with the plain 16-bit entry's on the same context.  The device
entries write between guard elements of 0xFFFF that must survive (the helpers of test_gpu_runner_up.py,
test_gpu_subpixel.py and test_gpu_web16.py)."""
import numpy as np
import pytest

import stereomatching_b200 as smb
import test_gpu_subpixel
from extras_model import reference_all
from test_gpu_flavours import FLAVOURS, assert_shape, code, diff, expected_shape, run_dev_batch
from test_gpu_min_shift import image_pair
from test_gpu_runner_up import run_dev as run_ru
from test_gpu_subpixel import run_dev as run_sub
from test_gpu_web16 import run16
from util import THRESHOLD, vname

pytestmark = pytest.mark.gpu

VARIANTS = [smb.WRAP, smb.GHOST]
FAMS = ("ru", "sub")
EXTRA = {"ru": 2, "sub": 3}  # each family's own output in reference_all's (best, web, runner_up, web_sub)
HOST_KW = {"ru": {"want_runner_up": True}, "sub": {"want_subpixel": True}}


@pytest.fixture(scope="module")
def num_sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def dev(c, fam, les, res, with_best=True, rows=None):
    """sm_match_wta_dev_batch_ru16 / _sub16 through the guarded helpers: (best or None, web, extra), (n, H, W)."""
    return (run_ru if fam == "ru" else run_sub)(c, les, res, with_best, rows)


def check(fam, got, refs, what, g16=None, rows=None):
    """got = (best or None, web, runner_up / web_sub) of n pairs against their reference_all tuples; g16 = the 16-bit
    entry's (best or None, web) on the same inputs and context; rows = (r0, r1) compares those rows only."""
    r0, r1 = rows if rows is not None else (0, got[1].shape[1])
    for k, ref in enumerate(refs):
        bo, wo, xo = (a[r0:r1] for a in (ref[0], ref[1], ref[EXTRA[fam]]))
        best, web, x = (None if a is None else np.asarray(a[k][r0:r1], np.int32) for a in got)
        w = "%s %s, pair %d" % (what, fam, k)
        if best is not None:
            assert np.array_equal(best, bo), "%s: best %s" % (w, diff(best, bo))
        assert np.array_equal(web, wo), "%s: web %s" % (w, diff(web, wo))
        assert np.array_equal(x, xo), "%s: %s %s" % (w, "runner_up" if fam == "ru" else "web_sub", diff(x, xo))
        if fam == "ru":
            assert (x <= bo).all(), w
        else:
            assert np.array_equal((x + 8) >> 4, web), w
        if g16 is not None:
            if best is not None and g16[0] is not None:
                assert np.array_equal(best, np.asarray(g16[0][k][r0:r1], np.int32)), w + ": best != the 16-bit entry's"
            assert np.array_equal(web, np.asarray(g16[1][k][r0:r1], np.int32)), w + ": web != the 16-bit entry's"


def inputs(W, H, D, m, seed):
    """(name, le, re): random maps at two densities whose second map is the first rolled by m + t (t in [0, D), a
    match inside the range) with 3 % flipped pixels, maps that never match (web == m + D everywhere), and, where the
    range holds one, maps periodic in x (ties between shifts a period apart)."""
    rng = np.random.default_rng(seed)
    out = []
    for dens in (0.15, 0.6):
        le = (rng.random((H, W)) < dens).astype(np.uint8)
        re = np.roll(le, m + int(rng.integers(0, D)), axis=1) ^ (rng.random((H, W)) < 0.03).astype(np.uint8)
        out.append(("random%.2f" % dens, le, re))
    out.append(("no_match", np.ones((H, W), np.uint8), np.zeros((H, W), np.uint8)))
    for P in (16, 32):
        if P < D and W % P == 0:
            le = np.tile((rng.random((H, P)) < 0.5).astype(np.uint8), (1, W // P))
            out.append(("periodic%d" % P, le, le.copy()))
            break
    return out


# ---------------------------------------------------------------------------------
# A. every shape family x m: one pair, several pairs, with and without best, a band
# ---------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
@pytest.mark.parametrize("flavour", list(FLAVOURS))
def test_shape_family(orc, num_sms, flavour, variant):
    nw, seg, multi, c2, hp, halves, geometry = FLAVOURS[flavour]
    half = halves[len(halves) // 2]
    W, H1, Hn, D = geometry(half, num_sms)
    sw = 2 * half + 1
    want = code(half, nw, seg, c2, hp, multi)
    one_pair = H1 <= 64  # (the one-word kernel's one-pair geometry has a CTA per SM: its batch geometry covers it)
    H = H1 if one_pair else Hn
    assert Hn is None or Hn == H
    for m in (1, 31, 33, 64, W - 1, W + 5, 2 * W + 3):
        tag = "%s half %d %dx%d D %d m %d %s" % (flavour, half, W, H, D, m, vname(variant))
        ins = inputs(W, H, D, m, 13 * m + W + D)
        refs = [reference_all(orc, name, le, re, D, sw, variant, m) for name, le, re in ins]
        if one_pair:
            with smb.StereoContext(W, H, D, sw, variant, kernel=smb.KERNEL_BITSLICE, min_shift=m) as c:
                for k, (name, le, re) in enumerate(ins):
                    g16 = run16(c, [le], [re])
                    assert_shape(c, want, "%s %s 16-bit" % (tag, name))
                    for fam in FAMS:
                        for with_best in (True, False) if k < 2 else (True,):
                            what = "%s %s one pair%s" % (tag, name, "" if with_best else ", no best")
                            got = dev(c, fam, [le], [re], with_best)
                            assert_shape(c, want, "%s %s" % (what, fam))
                            check(fam, got, refs[k:k + 1], what, g16)
        if Hn is not None:
            with smb.StereoContext(W, Hn, D, sw, variant, kernel=smb.KERNEL_BITSLICE, min_shift=m) as c:
                les, res = [f[1] for f in ins], [f[2] for f in ins]
                g16 = run16(c, les, res)
                assert_shape(c, want, tag + " 16-bit batch")
                for fam in FAMS:
                    for with_best in (True, False):
                        what = "%s, %d pairs per call%s" % (tag, len(ins), "" if with_best else ", no best")
                        got = dev(c, fam, les, res, with_best)
                        assert c.get_info(smb.INFO_PAIRS_PER_LAUNCH) >= len(ins), what + ": not one launch"
                        assert_shape(c, want, "%s %s" % (what, fam))
                        check(fam, got, refs, what, g16)
        # a band context: rows [r0, r1) only, the others keep their guard value
        r0, r1 = H // 3, H // 3 + max(1, min(H // 3, 20))
        band = expected_shape(W, r1 - r0, D, half, 1, num_sms)
        name, le, re = ins[1]
        with smb.StereoContext(W, H, D, sw, variant, rows=(r0, r1), kernel=smb.KERNEL_BITSLICE, min_shift=m) as c:
            g16 = run16(c, [le], [re], rows=(r0, r1))
            for fam in FAMS:
                what = "%s %s band [%d, %d)" % (tag, name, r0, r1)
                got = dev(c, fam, [le], [re], True, rows=(r0, r1))
                assert_shape(c, band, "%s %s" % (what, fam))
                check(fam, got, refs[1:2], what, g16, rows=(r0, r1))


# ---------------------------------------------------------------------------------
# B. more than 64 shifts, m > 0: winners on both sides of every chunk boundary
# ---------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
@pytest.mark.parametrize("D", [65, 129, 256])
def test_chunk_boundaries(orc, variant, D):
    """Right maps rolled by m + t for t on both sides of every 64-shift chunk boundary and at both range ends, and
    maps periodic in x that tie across the boundaries; one pair per launch and all of them in one launch."""
    W, H, sw = 384, 24, 9  # W > m + D: a WRAP roll has one best shift
    want = code(sw // 2, 2, 16, multi=True)
    half = sw // 2
    for m in (5, 37, 100):
        rng = np.random.default_rng(1000 * D + 10 * m + variant)
        ts = sorted({t for t in (0, 63, 64, 127, 128, D - 1) if t < D})
        ins = []
        for t in ts:
            le = (rng.random((H, W)) < 0.5).astype(np.uint8)
            flips = (rng.random((H, W)) < 0.03).astype(np.uint8)
            ins.append(("winners on %d" % t, le, np.roll(le, m + t, axis=1) ^ flips))
        for P in (16, 32, 64):
            le = np.tile((rng.random((H, P)) < 0.5).astype(np.uint8), (1, W // P))
            ins.append(("periodic%d" % P, le, le.copy()))
        refs = [reference_all(orc, "random", le, re, D, sw, variant, m) for _, le, re in ins]
        les, res = [f[1] for f in ins], [f[2] for f in ins]
        tag = "D %d m %d %s" % (D, m, vname(variant))
        with smb.StereoContext(W, H, D, sw, variant, min_shift=m) as c:
            g16 = run16(c, les, res)
            for fam in FAMS:
                for k, (name, le, re) in enumerate(ins):
                    got = dev(c, fam, [le], [re])
                    assert_shape(c, want, "%s %s one pair %s" % (tag, name, fam))
                    check(fam, got, refs[k:k + 1], "%s %s one pair" % (tag, name))
                for with_best in (True, False):
                    what = "%s batch%s" % (tag, "" if with_best else ", no best")
                    got = dev(c, fam, les, res, with_best)
                    assert_shape(c, want, "%s %s" % (what, fam))
                    check(fam, got, refs, what, g16)
        # the inputs do what the test is about, so that it cannot pass on zeros
        xs = np.arange(W)[None, :]
        for k, t in enumerate(ts):
            _, web, _, ws = refs[k]
            on = web == m + t + 1
            inside = np.ones((H, W), bool) if variant == smb.WRAP else np.broadcast_to(xs < W - m - t - half, (H, W))
            assert on[inside].mean() > 0.5, (tag, t)
            if 0 < t < D - 1:
                assert (ws[on] % 16 != 0).mean() > 0.3, (tag, t)
            else:
                assert (ws[on] == 16 * (m + t + 1)).all(), (tag, t)
        if variant == smb.WRAP:
            for k in (len(ts), len(ts) + 1):  # periods 16 and 32: every pixel ties across the chunks
                assert (refs[k][2] == refs[k][0]).mean() > 0.5, (tag, ins[k][0])


# ---------------------------------------------------------------------------------
# C. the direct kernel's twins with m > 0: forced, and the windows the auto kernel sends there
# ---------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
@pytest.mark.parametrize("W,H,D,sw,kernel", [(64, 40, 50, 9, smb.KERNEL_DIRECT), (64, 40, 130, 9, smb.KERNEL_DIRECT),
                                             (70, 66, 20, 33, smb.KERNEL_AUTO), (70, 66, 20, 45, smb.KERNEL_AUTO),
                                             (70, 66, 20, 63, smb.KERNEL_AUTO)],
                         ids=["forced_D50", "forced_D130", "window33", "window45", "window63"])
def test_direct_twins(orc, variant, W, H, D, sw, kernel):
    for m in (7, W + 3):
        tag = "%dx%d D %d window %d m %d %s" % (W, H, D, sw, m, vname(variant))
        ins = inputs(W, H, D, m, 17 * m + sw + D)[:3]
        refs = [reference_all(orc, name, le, re, D, sw, variant, m) for name, le, re in ins]
        les, res = [f[1] for f in ins], [f[2] for f in ins]
        with smb.StereoContext(W, H, D, sw, variant, kernel=kernel, min_shift=m) as c:
            g16 = run16(c, les, res, with_best=False)
            for fam in FAMS:
                got = dev(c, fam, les[:1], res[:1])
                assert_shape(c, smb.SHAPE_DIRECT, "%s one pair %s" % (tag, fam))
                check(fam, got, refs[:1], tag + " one pair")
                for with_best in (True, False):
                    got = dev(c, fam, les, res, with_best)
                    assert_shape(c, smb.SHAPE_DIRECT, "%s %s" % (tag, fam))
                    check(fam, got, refs, "%s, best %s" % (tag, with_best), g16)


# ---------------------------------------------------------------------------------
# D. the top of each family's range
# ---------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
@pytest.mark.parametrize("kernel", [smb.KERNEL_AUTO, smb.KERNEL_DIRECT], ids=["auto", "direct"])
def test_top_of_the_range(orc, variant, kernel):
    """web_sub at m + D == 4095, the runner-up and the 16-bit results at m + D == 65535, u8 webs at m + D == 255."""
    W, H, sw = 64, 24, 9
    for fam, top, Ds in (("sub", 4095, (65, 129)), ("ru", 65535, (1, 70))):
        for D in Ds:
            m = top - D
            tag = "D %d m %d %s" % (D, m, vname(variant))
            ins = inputs(W, H, D, m, top + D + variant)[:3]
            refs = [reference_all(orc, name, le, re, D, sw, variant, m) for name, le, re in ins]
            les, res = [f[1] for f in ins], [f[2] for f in ins]
            with smb.StereoContext(W, H, D, sw, variant, kernel=kernel, min_shift=m) as c:
                b16, w16 = run16(c, les, res)
                for k in range(len(ins)):
                    assert np.array_equal(b16[k], refs[k][0]) and np.array_equal(w16[k], refs[k][1]), (tag, "16-bit", k)
                for with_best in (True, False):
                    check(fam, dev(c, fam, les, res, with_best), refs, "%s, best %s" % (tag, with_best), (b16, w16))
                check(fam, dev(c, fam, les[:1], res[:1]), refs[:1], tag + " one pair", (b16, w16))
    for D in (1, 70):
        m = 255 - D
        tag = "u8 D %d m %d %s" % (D, m, vname(variant))
        name, le, re = inputs(W, H, D, m, 255 + D + variant)[1]
        bo, wo, _, _ = reference_all(orc, name, le, re, D, sw, variant, m)
        with smb.StereoContext(W, H, D, sw, variant, kernel=kernel, min_shift=m) as c:
            best, web = c.match_wta_host(le, re)
            assert np.array_equal(best, bo) and np.array_equal(web, wo), tag
            assert np.array_equal(c.download_web_u8(), wo.astype(np.uint8)), tag


# ---------------------------------------------------------------------------------
# E. the host-buffer entries from 8-bit images: batch, multi-GPU batch, bands
# ---------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
@pytest.mark.parametrize("W,H", [(128, 36), (67, 29)])  # (67 columns: the producers' generic kernels)
def test_host_entries(orc, variant, W, H):
    sw, n = 9, 5
    ndev = smb.device_count()
    devices = list(range(ndev)) if ndev > 1 else [0, 0, 0]  # (5 pairs over 3 slots: ragged shards)
    for D in (40, 100):
        for m in (3, 33, W + 5):
            tag = "%dx%d D %d m %d %s" % (W, H, D, m, vname(variant))
            pairs = [image_pair(orc, 4321 + 2 * k + m + D, W, H, m, D) for k in range(n)]
            first = np.stack([p[0] for p in pairs])
            second = np.stack([p[1] for p in pairs])
            refs = [reference_all(orc, "random", orc.edges(p[0], THRESHOLD, variant), orc.edges(p[1], THRESHOLD, variant),
                                  D, sw, variant, m) for p in pairs]
            with smb.StereoContext(W, H, D, sw, variant, min_shift=m) as c:
                c.set_option(smb.OPT_PIPE_GROUP, 2)  # several stages, a ragged last one
                w16, b16 = c.run_batch(first, second, THRESHOLD, want_best=True, web16=True)
                for fam in FAMS:
                    web, best, x = c.run_batch(first, second, THRESHOLD, want_best=True, web16=True, **HOST_KW[fam])
                    check(fam, (best, web, x), refs, tag + " run_batch", (b16, w16))
                    web, x = c.run_batch(first, second, THRESHOLD, web16=True, **HOST_KW[fam])
                    check(fam, (None, web, x), refs, tag + " run_batch, no best", (b16, w16))
            with smb.MultiGpuBatch(devices, W, H, D, sw, variant, min_shift=m) as mb:
                for fam in FAMS:
                    web, best, x = mb.run_batch(first, second, THRESHOLD, want_best=True, web16=True, **HOST_KW[fam])
                    check(fam, (best, web, x), refs, "%s multi %s" % (tag, devices), (b16, w16))
            for nb in (1, 2, 3):
                with smb.MultiGpuBands([0] * nb, W, H, D, sw, variant, min_shift=m) as bands:
                    for fam in FAMS:
                        web, best, x = bands.run(first[0], second[0], THRESHOLD, want_best=True, web16=True,
                                                 **HOST_KW[fam])
                        check(fam, (best[None], web[None], x[None]), refs[:1], "%s %d bands" % (tag, nb),
                              (b16[:1], w16[:1]))


# ---------------------------------------------------------------------------------
# F. one context, every family in sequence
# ---------------------------------------------------------------------------------
# D 100 at window 13: the MULTI runner-up and sub-pixel kernels hold 3 CTAs per SM, the int32 / 16-bit ones 4, so
# their launches take fewer pairs.  That shows in the launch counts only on a frame wide enough for a launch of
# fewer than 16 pairs to fill the machine three times over: 480 strips of 32 columns, one run of rows.
F_W, F_H, F_D, F_SW, F_M = 15360, 16, 100, 13, 21


def f_inputs(orc, variant, n, distinct=4):
    """n pairs of edge maps (distinct ones cycled) and their references."""
    rng = np.random.default_rng(600 + variant)
    les, res = [], []
    for k in range(distinct):
        le = (rng.random((F_H, F_W)) < 0.2 + 0.15 * k).astype(np.uint8)
        les.append(le)
        res.append(np.roll(le, F_M + 20 * k + 3, axis=1) ^ (rng.random((F_H, F_W)) < 0.03).astype(np.uint8))
    refs = [reference_all(orc, "random", le, re, F_D, F_SW, variant, F_M) for le, re in zip(les, res)]
    idx = [k % distinct for k in range(n)]
    return [les[i] for i in idx], [res[i] for i in idx], [refs[i] for i in idx]


@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
def test_one_context_every_family_dev(orc, monkeypatch, variant):
    n, few = 37, 13
    les, res, refs = f_inputs(orc, variant, n)

    def i32(c, k=n):
        best, web = run_dev_batch(c, les[:k], res[:k])
        for j in range(k):
            assert np.array_equal(best[j], refs[j][0]) and np.array_equal(web[j], refs[j][1]), ("i32", j)

    def u16(c, k=n):
        _, web = run16(c, les[:k], res[:k], with_best=False)
        for j in range(k):
            assert np.array_equal(web[j], refs[j][1]), ("u16", j)

    def fam_call(fam, with_best, k=n, guard=None):
        def call(c):
            with monkeypatch.context() as mp:
                if guard is not None:  # the helper's pairs lie out_stride = H*W + GUARD elements apart
                    mp.setattr(test_gpu_subpixel, "GUARD", guard)
                check(fam, dev(c, fam, les[:k], res[:k], with_best), refs[:k], "%s %d pairs" % (fam, k))
        return call

    steps = [("i32", i32), ("u16 without best", u16), ("ru16", fam_call("ru", True)),
             ("sub16 without best", fam_call("sub", False)),
             ("sub16 without best, larger out_stride", fam_call("sub", False, guard=3 * F_W + 5)),
             ("ru16 fewer pairs, without best", fam_call("ru", False, k=few)), ("i32 again", i32)]
    fresh = {}
    for name, step in steps:
        with smb.StereoContext(F_W, F_H, F_D, F_SW, variant, min_shift=F_M) as c:
            step(c)
            fresh[name] = c.last_launches()
    # the geometry is what the test is about: the runner-up / sub-pixel launches take fewer pairs than the int32 ones
    assert fresh["ru16"] > fresh["i32"] and fresh["sub16 without best"] > fresh["i32"], fresh
    with smb.StereoContext(F_W, F_H, F_D, F_SW, variant, min_shift=F_M) as c:
        for name, step in steps:
            step(c)
            assert c.last_launches() == fresh[name], "%s after the others: %d launches, %d on a fresh context" % (
                name, c.last_launches(), fresh[name])


@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
def test_one_context_every_family_host(orc, variant):
    n, few = 29, 7  # (a pipeline stage holds 16 pairs: a ragged last stage of 13, one launch or two)
    distinct = 3
    pairs = [image_pair(orc, 700 + 2 * k + variant, F_W, F_H, F_M, F_D) for k in range(distinct)]
    refs = [reference_all(orc, "random", orc.edges(p[0], THRESHOLD, variant), orc.edges(p[1], THRESHOLD, variant), F_D,
                          F_SW, variant, F_M) for p in pairs]
    refs = [refs[k % distinct] for k in range(n)]
    first = np.stack([pairs[k % distinct][0] for k in range(n)])
    second = np.stack([pairs[k % distinct][1] for k in range(n)])

    def plain(**kw):
        def call(c):
            web, best = c.run_batch(first, second, THRESHOLD, want_best=True, **kw)
            for j in range(n):
                assert np.array_equal(best[j].astype(np.int32), refs[j][0]), (kw, j)
                assert np.array_equal(web[j].astype(np.int32), refs[j][1]), (kw, j)
        return call

    def u8(c):
        web = c.run_batch(first, second, THRESHOLD, web_u8=True)
        for j in range(n):
            assert np.array_equal(web[j], refs[j][1].astype(np.uint8)), ("u8", j)

    def u16(c):
        web = c.run_batch(first, second, THRESHOLD, web16=True)
        for j in range(n):
            assert np.array_equal(web[j].astype(np.int32), refs[j][1]), ("u16", j)

    def fam_call(fam, with_best, k=n):
        def call(c):
            out = c.run_batch(first[:k], second[:k], THRESHOLD, want_best=with_best, web16=True, **HOST_KW[fam])
            got = (out[1], out[0], out[2]) if with_best else (None, out[0], out[1])
            check(fam, got, refs[:k], "run_batch %s %d pairs" % (fam, k))
        return call

    steps = [("i32", plain()), ("u16 without best", u16), ("ru16", fam_call("ru", True)),
             ("sub16 without best", fam_call("sub", False)), ("u8", u8), ("sub16", fam_call("sub", True)),
             ("ru16 fewer pairs, without best", fam_call("ru", False, k=few)), ("i32 again", plain())]
    fresh = {}
    for name, step in steps:
        with smb.StereoContext(F_W, F_H, F_D, F_SW, variant, min_shift=F_M) as c:
            step(c)
            fresh[name] = c.last_launches()
    assert fresh["ru16"] > fresh["i32"] and fresh["sub16"] > fresh["i32"], fresh
    with smb.StereoContext(F_W, F_H, F_D, F_SW, variant, min_shift=F_M) as c:
        for name, step in steps:
            step(c)
            assert c.last_launches() == fresh[name], "%s after the others: %d launches, %d on a fresh context" % (
                name, c.last_launches(), fresh[name])


# ---------------------------------------------------------------------------------
# G. a seeded random sample
# ---------------------------------------------------------------------------------
def test_random_sample(orc):
    seed = 20261022
    rng = np.random.default_rng(seed)
    for case in range(60):
        W, H = int(rng.integers(9, 301)), int(rng.integers(5, 61))
        sw = int(rng.integers(1, min(W, H, 31) + 1))
        D = int(rng.choice([int(rng.integers(1, 17)), int(rng.integers(17, 65)), int(rng.integers(65, 301))]))
        m = int(rng.integers(0, 3 * W + 41))
        variant = int(rng.integers(0, 2))
        kernel = (smb.KERNEL_AUTO, smb.KERNEL_DIRECT)[int(rng.integers(0, 2))]
        fam = FAMS[int(rng.integers(0, 2))]
        host = bool(rng.integers(0, 2))
        rows = None
        if not host and rng.integers(0, 2):
            r0 = int(rng.integers(0, H))
            rows = (r0, int(rng.integers(r0 + 1, H + 1)))
        tag = "seed %d case %d: %dx%d sw %d D %d m %d %s %s %s %s rows %s" % (
            seed, case, W, H, sw, D, m, vname(variant), "direct" if kernel else "auto", fam, "host" if host else "dev",
            rows)
        with smb.StereoContext(W, H, D, sw, variant, rows=rows, kernel=kernel, min_shift=m) as c:
            if host:
                left, right, _ = image_pair(orc, seed + case, W, H, m, D)
                ref = reference_all(orc, "random", orc.edges(left, THRESHOLD, variant),
                                    orc.edges(right, THRESHOLD, variant), D, sw, variant, m)
                web, best, x = c.run_batch(left[None], right[None], THRESHOLD, want_best=True, web16=True,
                                           **HOST_KW[fam])
                w16, b16 = c.run_batch(left[None], right[None], THRESHOLD, want_best=True, web16=True)
                check(fam, (best, web, x), [ref], tag, (b16, w16))
            else:
                le = (rng.random((H, W)) < rng.uniform(0.1, 0.7)).astype(np.uint8)
                re = np.roll(le, m + int(rng.integers(0, D)), axis=1) ^ (rng.random((H, W)) < 0.05).astype(np.uint8)
                ref = reference_all(orc, "random", le, re, D, sw, variant, m)
                g16 = run16(c, [le], [re], rows=rows)
                check(fam, dev(c, fam, [le], [re], True, rows=rows), [ref], tag, g16, rows=rows)
