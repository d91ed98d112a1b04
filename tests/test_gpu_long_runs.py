"""Row runs of many blocks through every 16-bit, runner-up and sub-pixel kernel, in one-pair, batch and band launches.

The bit-sliced kernel gives each warp a run of output rows and works through it in blocks of RB rows (8 or 16): the
window-filling prologue and blocks, then one steady block after another, then possibly one ragged last block.  State
carries from one steady block to the next: the tensor-memory ring of window rows, the shared-memory ring of centre
matches (the runner-up and sub-pixel families' aligned ring holds two or three whole blocks and wraps only after
them), the running sums and, past 64 shifts, the earlier chunks' best, runner-up, web_sub and carry, prefetched per
block.  The other tests force the number of runs for the int32 family only, and their frames are short enough that
the cost model's runs hold about one block each.  Here every reachable instantiation runs a frame of 7 whole blocks
and a ragged one of 1 or RB - 1 rows (the one-word kernel one CTA per SM and more, to keep its 16-pixel segments),
with the runs forced through SM_OPT_ROW_RUNS: one run of the whole frame, 2, 3, one per block, a count above that
(clamped) and the cost model's.  The same frames then go through launches of several pairs and through row bands, and
the host entries run from 8-bit images with one run per frame.

Two inputs per kernel: the random pair of test_gpu_flavours.families, and a pair whose rows are shifted in bands of 5
rows (5 is coprime with 8 and 16, so band edges fall at every row of a block).  The bands' shifts include both ends of
the range and both sides of every 64-shift chunk boundary, so a ring slot off by a row or a block changes web there.
Every output is compared bit for bit with tests/extras_model.py, between guard elements that must survive."""
import functools

import numpy as np
import pytest

import stereomatching_b200 as smb
from extras_model import reference_all
from test_gpu_flavours import (FLAVOURS, REACHABLE, assert_shape, code, diff, expected_shape, families, row_runs_for,
                               rows_per_block, run_dev_batch)
from test_gpu_min_shift import image_pair
from test_gpu_range_extras import HOST_KW, check, dev
from test_gpu_web16 import run16
from util import THRESHOLD, vname

pytestmark = pytest.mark.gpu

VARIANTS = [smb.WRAP, smb.GHOST]
FAMS = ("ru", "sub")
SEG8 = {c for c in REACHABLE if c & smb.SHAPE_SEG8}
# launches of several pairs never take 8-pixel segments: the flavours they reach
BATCH_FLAVOURS = [f for f, v in FLAVOURS.items() if v[1] == 16]
# shape codes compared with the model: in one-pair launches of one run over the whole frame (at least
# ceil((RB + half + 1) / RB) + 2 steady blocks, more than either centre-match ring holds) ...
LONG = {"u16": set(), "ru": set(), "sub": set()}
# ... and in launches of several pairs, one run per pair
BATCH = {"i32": set(), "u16": set(), "ru": set(), "sub": set()}
DONE = set()  # parametrised cases of this file that completed


@pytest.fixture(scope="module")
def num_sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


# ---------------------------------------------------------------------------------
# geometries, inputs and references
# ---------------------------------------------------------------------------------
def tall(flavour, half, num_sms):
    """(W, H, D, m, RB, shape) of a flavour's tall one-pair frame: its width and shift count (so its kernel), 7 whole
    blocks and a ragged one (the one-word kernel: 16 * num_sms rows and a ragged block, one CTA per SM and more).  Even
    halves end on a block of one row, odd ones on RB - 1 rows.  half // 2 even searches from shift 0, odd from 37, or
    from 5 in frames under 100 columns (in GHOST a range from 37 leaves most of such a frame without a match)."""
    nw, seg, multi, c2, hp, _, geometry = FLAVOURS[flavour]
    W, _, _, D = geometry(half, num_sms)
    shape = code(half, nw, seg, c2, hp, multi)
    RB = rows_per_block(shape)
    r = 1 if half % 2 == 0 else RB - 1
    H = (16 * num_sms if flavour == "one_word" else 7 * RB) + r
    m = 0 if half // 2 % 2 == 0 else (37 if W >= 100 else 5)
    assert expected_shape(W, H, D, half, 1, num_sms) == shape, (flavour, half)
    return W, H, D, m, RB, shape


def banded(W, H, D, m, seed):
    """(le, re): row y of re is that of le rolled by the shift of band y // 5, then 3 % of the pixels flipped (so that
    fractions are not zero).  Even bands take in turn the range's first and last shift and both sides of each 64-shift
    chunk boundary (winners left pending across chunks), odd bands a random shift of the range."""
    rng = np.random.default_rng(seed)
    ends = sorted({m, m + D - 1} | {m + b + t for b in range(64, D, 64) for t in (-1, 0)})
    shifts = [ends[b // 2 % len(ends)] if b % 2 == 0 else int(rng.integers(m, m + D)) for b in range(-(-H // 5))]
    le = (rng.random((H, W)) < 0.5).astype(np.uint8)
    re = np.stack([np.roll(le[y], shifts[y // 5]) for y in range(H)])
    return le, re ^ (rng.random((H, W)) < 0.03).astype(np.uint8)


def assert_bands_bite(ref, D, m, what):
    """The banded input does its job: web changes down most columns, and many inner winners have a fraction."""
    _, web, _, ws = ref
    if D < 3:  # one web, or no inner winner
        return
    several = np.mean([len(np.unique(web[:, x])) >= 3 for x in range(web.shape[1])])
    assert several > 0.5, "%s: web takes 3 values or more in only %.2f of the columns" % (what, several)
    inner = (web > m + 1) & (web < m + D)
    frac = (ws[inner] % 16 != 0).mean()
    assert inner.mean() > 0.05 and frac > 0.3, "%s: %.2f inner winners, %.2f of them with a fraction" % (
        what, inner.mean(), frac)


@functools.lru_cache(maxsize=None)
def cases(orc, flavour, variant, num_sms):
    """Per half of the flavour: (half, W, H, D, m, RB, shape, inputs), inputs a list of (name, le, re, reference_all's
    (best, web, runner_up, web_sub)): the random pair, the banded pair and one more random pair for the batch."""
    out = []
    for half in FLAVOURS[flavour][5]:
        W, H, D, m, RB, shape = tall(flavour, half, num_sms)
        sw = 2 * half + 1
        seed = 3000 + 1000 * half + 17 * D + W + variant
        pairs = [("random", *families(W, H, D, seed)[1][1:]), ("banded", *banded(W, H, D, m, seed)),
                 ("random, second", *families(W, H, D, seed + 1)[1][1:])]
        ins = [(name, le, re, reference_all(orc, "random", le, re, D, sw, variant, m)) for name, le, re in pairs]
        assert_bands_bite(ins[1][3], D, m, "%s half %d %s" % (flavour, half, vname(variant)))
        out.append((half, W, H, D, m, RB, shape, ins))
    return out


# ---------------------------------------------------------------------------------
# checks
# ---------------------------------------------------------------------------------
def assert_runs(c, shape, BH, RB, runs, what):
    """The launch ran `shape` with the row runs asked for (0: the cost model's, at most one per block)."""
    assert_shape(c, shape, what)
    got = c.get_info(smb.INFO_ROW_RUNS)
    if runs:
        assert got == row_runs_for(BH, RB, runs)[0], "%s: %d row runs launched" % (what, got)
    else:
        assert 1 <= got <= -(-BH // RB), "%s: %d row runs launched" % (what, got)


def assert_one_launch(c, shape, BH, RB, runs, npairs, what):
    assert c.get_info(smb.INFO_PAIRS_PER_LAUNCH) >= npairs, what + ": the pairs do not fit one launch"
    assert c.last_launches() == 2, "%s: %d launches, not a pack and a main kernel" % (what, c.last_launches())
    assert_runs(c, shape, BH, RB, runs, what)


def check16(got, refs, what, rows=None):
    """(best or None, web) of n pairs, from the int32 or the 16-bit entry, against their reference_all tuples."""
    r0, r1 = rows if rows is not None else (0, got[1].shape[1])
    for k, ref in enumerate(refs):
        for name, a, want in (("best", got[0], ref[0]), ("web", got[1], ref[1])):
            if a is not None:
                a = np.asarray(a[k][r0:r1], np.int32)
                assert np.array_equal(a, want[r0:r1]), "%s, pair %d: %s %s" % (what, k, name, diff(a, want[r0:r1]))


# ---------------------------------------------------------------------------------
# one pair per launch, the row runs forced
# ---------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
@pytest.mark.parametrize("flavour", list(FLAVOURS))
def test_one_pair_long_runs(orc, num_sms, flavour, variant):
    for half, W, H, D, m, RB, shape, ins in cases(orc, flavour, variant, num_sms):
        sw = 2 * half + 1
        max_runs = -(-H // RB)
        # one run of the whole frame: H // RB steady blocks, then the ragged one
        assert H // RB >= -(-(RB + half + 1) // RB) + 2
        with smb.StereoContext(W, H, D, sw, variant, kernel=smb.KERNEL_BITSLICE, min_shift=m) as c:
            for name, le, re, ref in ins[:2]:
                for runs in (1, 2, 3, max_runs, 10 ** 6, 0):
                    c.set_option(smb.OPT_ROW_RUNS, runs)
                    for with_best in (True, False) if runs == 1 else (True,):
                        what = "%s half %d %dx%d D %d m %d %s %s, %d row runs asked%s" % (
                            flavour, half, W, H, D, m, vname(variant), name, runs, "" if with_best else ", no best")
                        g16 = run16(c, [le], [re], with_best)
                        assert_runs(c, shape, H, RB, runs, what + " 16-bit")
                        check16(g16, [ref], what + " 16-bit")
                        for fam in FAMS:
                            got = dev(c, fam, [le], [re], with_best)
                            assert_runs(c, shape, H, RB, runs, "%s %s" % (what, fam))
                            check(fam, got, [ref], what, g16)
                    if runs == 1:
                        for fam in LONG:
                            LONG[fam].add(shape)
    DONE.add(("one pair", flavour, variant))


# ---------------------------------------------------------------------------------
# several pairs in one launch, the row runs forced: the per-group scratch best and carry with long runs
# ---------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
@pytest.mark.parametrize("flavour", BATCH_FLAVOURS)
def test_batch_long_runs(orc, num_sms, flavour, variant):
    for half, W, H, D, m, RB, shape, ins in cases(orc, flavour, variant, num_sms):
        sw = 2 * half + 1
        les, res, refs = [i[1] for i in ins], [i[2] for i in ins], [i[3] for i in ins]
        n = len(ins)
        with smb.StereoContext(W, H, D, sw, variant, kernel=smb.KERNEL_BITSLICE, min_shift=m) as c:
            for runs in (1, 3):
                c.set_option(smb.OPT_ROW_RUNS, runs)
                tag = "%s half %d %dx%d D %d m %d %s, %d pairs, %d row runs asked" % (
                    flavour, half, W, H, D, m, vname(variant), n, runs)
                got = run_dev_batch(c, les, res)
                assert_one_launch(c, shape, H, RB, runs, n, tag + " int32")
                check16(got, refs, tag + " int32")
                for with_best in (True, False):
                    what = tag + ("" if with_best else ", no best")
                    g16 = run16(c, les, res, with_best)
                    assert_one_launch(c, shape, H, RB, runs, n, what + " 16-bit")
                    check16(g16, refs, what + " 16-bit")
                    for fam in FAMS:
                        got = dev(c, fam, les, res, with_best)
                        assert_one_launch(c, shape, H, RB, runs, n, "%s %s" % (what, fam))
                        check(fam, got, refs, what, g16)
                if runs == 1:
                    for fam in BATCH:
                        BATCH[fam].add(shape)
    DONE.add(("batch", flavour, variant))


# ---------------------------------------------------------------------------------
# row bands of 5 blocks and more, starting 3 rows into a block
# ---------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
@pytest.mark.parametrize("flavour", list(FLAVOURS))
def test_band_long_runs(orc, num_sms, flavour, variant):
    for half, W, H, D, m, RB, shape, ins in cases(orc, flavour, variant, num_sms):
        sw = 2 * half + 1
        nb = 5 * RB + 2
        band = expected_shape(W, nb, D, half, 1, num_sms)  # (a short one-word band takes 8-pixel segments)
        RBb = rows_per_block(band)
        r0 = RBb + 3
        r1 = r0 + nb
        assert r1 <= H
        with smb.StereoContext(W, H, D, sw, variant, rows=(r0, r1), kernel=smb.KERNEL_BITSLICE, min_shift=m) as c:
            for name, le, re, ref in ins[:2]:
                for runs in (1, 2):
                    c.set_option(smb.OPT_ROW_RUNS, runs)
                    what = "%s half %d %dx%d D %d m %d %s %s, band [%d, %d), %d row runs asked" % (
                        flavour, half, W, H, D, m, vname(variant), name, r0, r1, runs)
                    g16 = run16(c, [le], [re], rows=(r0, r1))
                    assert_runs(c, band, nb, RBb, runs, what + " 16-bit")
                    check16(g16, [ref], what + " 16-bit", rows=(r0, r1))
                    for fam in FAMS:
                        got = dev(c, fam, [le], [re], True, rows=(r0, r1))
                        assert_runs(c, band, nb, RBb, runs, "%s %s" % (what, fam))
                        check(fam, got, [ref], what, g16, rows=(r0, r1))
    DONE.add(("band", flavour, variant))


# ---------------------------------------------------------------------------------
# the host entries from 8-bit images: one run per frame, pipeline stages of 2 pairs (a ragged last one)
# ---------------------------------------------------------------------------------
HOST = [(200, 59, 129, 9, 5, code(4, 2, 16, multi=True)), (160, 61, 25, 11, 37, code(5, 2, 16, c2=True))]


@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
@pytest.mark.parametrize("W,H,D,sw,m,shape", HOST, ids=["two_words_chunks", "column_pairs"])
def test_host_long_runs(orc, variant, W, H, D, sw, m, shape):
    n = 5
    RB = rows_per_block(shape)
    tag = "%dx%d D %d window %d m %d %s, one row run asked" % (W, H, D, sw, m, vname(variant))
    pairs = [image_pair(orc, 5100 + 7 * k + m + D, W, H, m, D) for k in range(n)]
    first = np.stack([p[0] for p in pairs])
    second = np.stack([p[1] for p in pairs])
    refs = [reference_all(orc, "random", orc.edges(p[0], THRESHOLD, variant), orc.edges(p[1], THRESHOLD, variant), D,
                          sw, variant, m) for p in pairs]
    with smb.StereoContext(W, H, D, sw, variant, min_shift=m) as c:
        c.set_option(smb.OPT_PIPE_GROUP, 2)
        c.set_option(smb.OPT_ROW_RUNS, 1)
        w16, b16 = c.run_batch(first, second, THRESHOLD, want_best=True, web16=True)
        assert_runs(c, shape, H, RB, 1, tag + " 16-bit")
        check16((b16, w16), refs, tag + " run_batch 16-bit")
        for fam in FAMS:
            web, best, x = c.run_batch(first, second, THRESHOLD, want_best=True, web16=True, **HOST_KW[fam])
            assert_runs(c, shape, H, RB, 1, "%s %s" % (tag, fam))
            check(fam, (best, web, x), refs, tag + " run_batch", (b16, w16))
            web, x = c.run_batch(first, second, THRESHOLD, web16=True, **HOST_KW[fam])
            assert_runs(c, shape, H, RB, 1, "%s %s, no best" % (tag, fam))
            check(fam, (None, web, x), refs, tag + " run_batch, no best", (b16, w16))
    DONE.add(("host", W, variant))


def test_every_reachable_kernel_ran_long_runs():
    """Runs last: every reachable 16-bit, runner-up and sub-pixel kernel was compared with the model in a run of many
    steady blocks, and every one a launch of several pairs can take in all four families."""
    cases_in_file = 2 * (2 * len(FLAVOURS) + len(BATCH_FLAVOURS) + len(HOST))
    if len(DONE) < cases_in_file:
        pytest.skip("needs every parametrised case of this file to have passed in this session")
    assert len(REACHABLE) == 87 and len(SEG8) == 16
    for seen, want in [(LONG, REACHABLE), (BATCH, REACHABLE - SEG8)]:
        for fam, codes in seen.items():
            assert codes == want, "%s: missing %s, unexpected %s" % (
                fam, sorted(hex(x) for x in want - codes), sorted(hex(x) for x in codes - want))
