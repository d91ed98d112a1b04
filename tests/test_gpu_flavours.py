"""Every instantiation of the bit-sliced kernel against the oracle, in one-pair and several-pairs launches.

k_bitslice is a family of template instantiations <HALF, NW, SEG, MULTI, C2, HP>; pick_shape / launch_one choose one
from the window half, the shift count, the frame width, the band height, the pairs per launch and the SM count.
Each launch reports what it ran (SM_INFO_KERNEL_SHAPE, SM_INFO_ROW_RUNS), so the tests below assert which kernel
they compared, and the last test asserts that the table of reachable kernels was launched in full.

Per kernel and variant the inputs are: random maps at two densities; saturated maps (le == re == 0: every shift
matches, the box count reaches (2h+1)^2, the top of its bit planes, and every shift ties); maps that never match
(le = 1, re = 0: all scores 0, web == num_shifts); and maps periodic in x (re == le, period P < num_shifts), whose
full-window ties at 0, P, 2P, ... sit on lane, word and chunk boundaries.  Then the row runs of a one-pair launch,
several distinct pairs in one launch, and two row bands (one shorter than a block and than 2*half, one ending at the
frame's last row).  Separate tests cover a ragged batch whose last launch has one pair, and frames on both sides of
every selection switch.
"""
import numpy as np
import pytest

import stereomatching_b200 as smb
from util import THRESHOLD, vname

pytestmark = pytest.mark.gpu

VARIANTS = [smb.WRAP, smb.GHOST]


def code(half, nw, seg, c2=False, hp=False, multi=False):
    """The SM_INFO_KERNEL_SHAPE code of k_bitslice<half, nw, seg, multi, c2, hp>."""
    return (smb.SHAPE_BITSLICE | half | (smb.SHAPE_TWO_WORDS if nw == 2 else 0) | (smb.SHAPE_SEG8 if seg == 8 else 0)
            | (smb.SHAPE_C2 if c2 else 0) | (smb.SHAPE_HP if hp else 0) | (smb.SHAPE_MULTI if multi else 0))


def rows_per_block(shape):
    return 8 if shape & (smb.SHAPE_TWO_WORDS | smb.SHAPE_SEG8) else 16


def expected_shape(W, BH, D, half, npairs, num_sms):
    """The kernel the release library picks for a launch (pick_shape in k_bitslice.cu), for the selection tests."""
    seg, hp = 16, False
    if D > 32:
        nw, c2 = 2, False
    else:
        c2 = W >= 64 and half <= 6
        nw = 2 if c2 else 1
        hp = D <= 16 and W >= 64
        if nw == 1 and not hp and npairs == 1:
            ctas = ((W + 31) // 32 + 3) // 4 * ((BH + 15) // 16)
            if ctas < num_sms:
                seg = 8
    return code(half, nw, seg, c2, hp, multi=not c2 and nw == 2 and D > 64)


def row_runs_for(BH, RB, want):
    """(runs, rows per run) of a launch asked for `want` runs: whole blocks of RB rows per run (shape() in
    launch_one); the last run has the rows left over."""
    sg = min(max(want, 1), -(-BH // RB))
    rows = -(-BH // sg)
    rows = -(-rows // RB) * RB
    return -(-BH // rows), rows


# ---------------------------------------------------------------------------------
# the flavour table: the 87 instantiations the release build can launch
# ---------------------------------------------------------------------------------
# name -> (NW, SEG, MULTI, C2, HP, halves, geometry(half, num_sms) -> (W, H one pair, H several pairs or None, D))
FLAVOURS = {
    # 32 shifts or fewer, frames under 64 columns: one word per lane.  A one-pair launch keeps 16-pixel segments only
    # when the frame has at least one CTA per SM (48 columns are one CTA per 16 rows: 16 * num_sms rows)
    "one_word": (1, 16, False, False, False, range(16),
                 lambda h, n: (48, 16 * n, 40, (30, 32, 17, 25)[h % 4])),
    # the same kernel with 8-pixel segments: one pair per launch, under one CTA per SM.  A launch of several pairs
    # never takes it (test_ragged_batch_ends_on_the_small_frame_kernel covers a batch's one-pair last launch)
    "one_word_seg8": (1, 8, False, False, False, range(16),
                      lambda h, n: (48, 40, None, (30, 32, 17, 25)[h % 4])),
    # 33..64 shifts: two shift words per lane
    "two_words": (2, 16, False, False, False, range(16),
                  lambda h, n: (64, 40, 40, (50, 33, 64, 47)[h % 4])),
    # more than 64 shifts: 64-shift chunks merged in place
    "two_words_chunks": (2, 16, True, False, False, range(16),
                         lambda h, n: (64, 40, 40, (100, 70, 129)[h % 3])),
    # 16 shifts or fewer, at least 64 columns, windows 15 and up: two pixels per word
    "half_word_pairs": (1, 16, False, False, True, range(7, 16),
                        lambda h, n: (100, 40, 40, (16, 13, 9)[h % 3])),
    # 17..32 shifts, at least 64 columns, windows up to 13: the two words of a lane are two pixels
    "column_pairs": (2, 16, False, True, False, range(7),
                     lambda h, n: (128, 40, 40, (30, 32, 17, 25)[h % 4])),
    # 16 shifts or fewer, at least 64 columns, windows up to 13: both
    "column_half_word_pairs": (2, 16, False, True, True, range(7),
                               lambda h, n: (160, 40, 40, (16, 9, 1, 13)[h % 4])),
}
REACHABLE = {code(h, nw, seg, c2, hp, multi)
             for nw, seg, multi, c2, hp, halves, _ in FLAVOURS.values() for h in halves}
# k_bitslice<h, 1, 16, false, false, true> for halves 0..6 is compiled and listed in dispatch(), but the release build
# never picks it: half-word pairs need at least 64 columns, and at 64 columns or more windows up to 13 take column
# pairs.  Only the development build's SMB_NO_C2 switch reaches it.
UNREACHABLE = {code(h, 1, 16, hp=True) for h in range(7)}

SEEN = set()  # codes of the launches the flavour table compared with the oracle
DONE = set()  # (flavour, variant) tests that completed


@pytest.fixture(scope="module")
def num_sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


# ---------------------------------------------------------------------------------
# inputs and the oracle
# ---------------------------------------------------------------------------------
def families(W, H, D, seed):
    """(name, le, re) inputs for one geometry."""
    rng = np.random.default_rng(seed)
    out = []
    for dens in (0.15, 0.6):
        le = (rng.random((H, W)) < dens).astype(np.uint8)
        re = np.roll(le, int(rng.integers(0, min(D, W))), axis=1) ^ (rng.random((H, W)) < 0.03).astype(np.uint8)
        out.append(("random%.2f" % dens, le, re))
    out.append(("saturated", np.zeros((H, W), np.uint8), np.zeros((H, W), np.uint8)))
    out.append(("no_match", np.ones((H, W), np.uint8), np.zeros((H, W), np.uint8)))
    for P in (16, 32, 64):
        if P < D and W % P == 0:
            le = np.tile((rng.random((H, P)) < 0.5).astype(np.uint8), (1, W // P))
            out.append(("periodic%d" % P, le, le.copy()))
    return out


def reference(orc, name, le, re, D, sw, variant):
    """The oracle's (best, web).  The literal sw*sw tap loop for saturated maps and small problems, the separable
    sums otherwise.  Maps whose rows are all equal are evaluated on 2*half+1 rows: every output row of the frame
    then equals the row of that small frame with the same rows of the window inside the frame (all of them in
    WRAP; the first and last `half` rows differ in GHOST)."""
    H, W = le.shape
    half = sw // 2
    N = 2 * half + 1
    if H > N and (le == le[:1]).all() and (re == re[:1]).all():
        b, w = reference(orc, name, le[:N], re[:N], D, sw, variant)
        ys = np.arange(H)
        src = np.where(ys < half, ys, np.where(ys >= H - half, ys - (H - N), half))
        return b[src], w[src]
    direct = name == "saturated" or W * H * D * N * N <= 10 ** 6
    return orc.match_wta(le, re, D, sw, variant, direct=direct)


def diff(got, want):
    bad = np.argwhere(got != want)
    return "%d pixels differ, first (y, x) %s: %s != %s" % (
        len(bad), tuple(bad[0]), got[tuple(bad[0])], want[tuple(bad[0])]) if len(bad) else "equal"


def assert_equal(best, web, bo, wo, what):
    assert np.array_equal(best, bo), "%s: best %s" % (what, diff(best, bo))
    assert np.array_equal(web, wo), "%s: web %s" % (what, diff(web, wo))


def assert_shape(c, want, what, record=None):
    got = c.get_info(smb.INFO_KERNEL_SHAPE)
    assert got == want, "%s: launched shape %#x, expected %#x" % (what, got, want)
    if record is not None:
        record.add(got)


def run_dev_batch(c, les, res):
    """sm_match_wta_dev_batch over distinct pairs; returns (best, web) as (n, H, W) arrays."""
    import torch
    n, (H, W) = len(les), les[0].shape
    d1 = torch.from_numpy(np.stack(les)).cuda()
    d2 = torch.from_numpy(np.stack(res)).cuda()
    best = torch.full((n, H, W), -7, dtype=torch.int32, device="cuda")
    web = torch.full((n, H, W), -7, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    c.match_wta_dev_batch(n, d1.data_ptr(), d2.data_ptr(), H * W, best.data_ptr(), web.data_ptr(), H * W)
    c.synchronize()
    return best.cpu().numpy(), web.cpu().numpy()


# ---------------------------------------------------------------------------------
# the table
# ---------------------------------------------------------------------------------
def test_flavour_table_is_complete():
    assert len(REACHABLE) == 87 and len(UNREACHABLE) == 7 and not REACHABLE & UNREACHABLE


@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
@pytest.mark.parametrize("flavour", list(FLAVOURS))
def test_flavour(orc, num_sms, flavour, variant):
    nw, seg, multi, c2, hp, halves, geometry = FLAVOURS[flavour]
    for half in halves:
        want = code(half, nw, seg, c2, hp, multi)
        RB = rows_per_block(want)
        W, H1, Hn, D = geometry(half, num_sms)
        sw = 2 * half + 1
        seed = 1000 * half + 17 * D + W
        tag = "%s half %d %dx%d D %d %s" % (flavour, half, W, H1, D, vname(variant))
        fams1 = fams = families(W, H1, D, seed)
        refs1 = refs = {name: reference(orc, name, le, re, D, sw, variant) for name, le, re in fams}
        with smb.StereoContext(W, H1, D, sw, variant, kernel=smb.KERNEL_BITSLICE) as c:
            assert c.get_info(smb.INFO_KERNEL_SHAPE) == 0 and c.get_info(smb.INFO_ROW_RUNS) == 0
            # one pair per launch, every input family
            for name, le, re in fams:
                best, web = c.match_wta_host(le, re)
                assert_shape(c, want, "%s %s" % (tag, name), SEEN)
                assert_equal(best, web, *refs[name], "%s %s" % (tag, name))
            # row runs: the cost model's, one, two, the most the frame allows, and a count with a ragged last run
            name, le, re = fams[1]
            max_runs = -(-H1 // RB)
            ragged = [r for r in range(3, max_runs + 1) if H1 % row_runs_for(H1, RB, r)[1]]
            for runs in [0, 1, 2, max_runs] + ragged[:1]:
                c.set_option(smb.OPT_ROW_RUNS, runs)
                best, web = c.match_wta_host(le, re)
                what = "%s %s, %d row runs asked" % (tag, name, runs)
                assert_shape(c, want, what)
                got = c.get_info(smb.INFO_ROW_RUNS)
                if runs:
                    assert got == row_runs_for(H1, RB, runs)[0], "%s: %d launched" % (what, got)
                else:
                    assert 1 <= got <= max_runs, "%s: %d launched" % (what, got)
                assert_equal(best, web, *refs[name], what)
            c.set_option(smb.OPT_ROW_RUNS, 0)
        # several distinct pairs in one launch (the throughput shape); every family is one pair of the batch
        if Hn is not None:
            if Hn != H1:
                fams = families(W, Hn, D, seed + 1)
                refs = {name: reference(orc, name, le, re, D, sw, variant) for name, le, re in fams}
            with smb.StereoContext(W, Hn, D, sw, variant, kernel=smb.KERNEL_BITSLICE) as c:
                best, web = run_dev_batch(c, [f[1] for f in fams], [f[2] for f in fams])
                what = "%s, %d pairs per call" % (tag, len(fams))
                assert c.get_info(smb.INFO_PAIRS_PER_LAUNCH) >= len(fams), what + ": not one launch"
                assert_shape(c, want, what, SEEN)
                for k, (name, _, _) in enumerate(fams):
                    assert_equal(best[k], web[k], *refs[name], "%s, pair %d (%s)" % (what, k, name))
        # row bands of the one-pair frame: one shorter than a block and than 2*half in the middle, one ending at the
        # last row.  A band's height selects its own kernel (a short one-word band takes 8-pixel segments)
        name, le, re = fams1[1]
        bo, wo = refs1[name]
        short = max(1, min(RB, 2 * half) - 1)
        for r0, r1 in [(H1 // 2 - short // 2, H1 // 2 - short // 2 + short), (H1 - min(H1 - 1, RB + half + 3), H1)]:
            what = "%s %s, band rows [%d, %d)" % (tag, name, r0, r1)
            with smb.StereoContext(W, H1, D, sw, variant, rows=(r0, r1), kernel=smb.KERNEL_BITSLICE) as c:
                c.set_edges(le, re)
                c.match_wta()
                best = c.download(smb.BEST, out=np.full((H1, W), -7, np.int32))
                web = c.download(smb.WEB, out=np.full((H1, W), -7, np.int32))
                assert_shape(c, expected_shape(W, r1 - r0, D, half, 1, num_sms), what)
            assert_equal(best[r0:r1], web[r0:r1], bo[r0:r1], wo[r0:r1], what)
    DONE.add((flavour, variant))


@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
def test_ragged_batch_ends_on_the_small_frame_kernel(orc, num_sms, variant):
    """17 pairs of a small one-word frame: one launch of 16 pairs, then one of a single pair, which takes the
    8-pixel-segment kernel and the one-pair launch shape.  Through the device-pointer batch and sm_run_batch."""
    n, W, H, D, sw = 17, 48, 40, 30, 21
    small = code(sw // 2, 1, 8)
    rng = np.random.default_rng(17 + variant)
    les = [(rng.random((H, W)) < (0.1 + 0.05 * k)).astype(np.uint8) for k in range(n)]
    res = [np.roll(le, k % D, axis=1) ^ (rng.random((H, W)) < 0.02).astype(np.uint8) for k, le in enumerate(les)]
    with smb.StereoContext(W, H, D, sw, variant) as c:
        best, web = run_dev_batch(c, les, res)
        assert c.get_info(smb.INFO_PAIRS_PER_LAUNCH) == 16
        assert_shape(c, small, "sm_match_wta_dev_batch, last launch", SEEN)
    for k in range(n):
        assert_equal(best[k], web[k], *reference(orc, "random", les[k], res[k], D, sw, variant), "dev batch pair %d" % k)
    pairs = [orc.synth_pair(600 + 2 * k, W, H, D) for k in range(n)]
    first, second = np.stack([p[0] for p in pairs]), np.stack([p[1] for p in pairs])
    with smb.StereoContext(W, H, D, sw, variant) as c:
        web, best = c.run_batch(first, second, THRESHOLD, want_best=True)
        assert_shape(c, small, "sm_run_batch, last launch", SEEN)
    for k in range(n):
        e1, e2 = orc.edges(first[k], THRESHOLD, variant), orc.edges(second[k], THRESHOLD, variant)
        assert_equal(best[k], web[k], *reference(orc, "random", e1, e2, D, sw, variant), "run_batch pair %d" % k)


@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
def test_selection_boundaries(orc, num_sms, variant):
    """Frames on both sides of every switch of the kernel selection: column pairs from 64 columns and up to window
    13, the 64-column strips of half-word pairs and 128-column strips of column + half-word pairs, and the 8-pixel
    segments of one-pair launches below one CTA per SM (16-row blocks, one CTA per block row at 48 columns)."""
    n = num_sms
    cases = [(w, 40, 30, h) for h in (2, 6, 7) for w in (63, 64, 65)]
    cases += [(w, 40, 16, h) for h in (3, 9) for w in (63, 64, 65, 127, 128, 129)]
    cases += [(48, H, 30, 4) for H in (16 * (n - 1), 16 * (n - 1) + 1, 16 * n)]
    seen = set()
    for (W, H, D, half) in cases:
        sw = 2 * half + 1
        rng = np.random.default_rng(W * 1000 + H + half)
        les = [(rng.random((H, W)) < d).astype(np.uint8) for d in (0.2, 0.5, 0.8)]
        res = [np.roll(le, k + 3, axis=1) ^ (rng.random((H, W)) < 0.03).astype(np.uint8) for k, le in enumerate(les)]
        refs = [reference(orc, "random", le, re, D, sw, variant) for le, re in zip(les, res)]
        tag = "%dx%d D %d half %d" % (W, H, D, half)
        with smb.StereoContext(W, H, D, sw, variant) as c:
            best, web = c.match_wta_host(les[0], res[0])
            assert_shape(c, expected_shape(W, H, D, half, 1, n), tag + ", one pair", seen)
            assert_equal(best, web, *refs[0], tag + ", one pair")
            best, web = run_dev_batch(c, les, res)
            assert_shape(c, expected_shape(W, H, D, half, 3, n), tag + ", three pairs", seen)
            for k in range(3):
                assert_equal(best[k], web[k], *refs[k], "%s, three pairs, pair %d" % (tag, k))
    # each switch was seen from both sides
    assert code(6, 2, 16, c2=True) in seen and code(6, 1, 8) in seen and code(7, 1, 8) in seen
    assert code(3, 2, 16, c2=True, hp=True) in seen and code(9, 1, 16, hp=True) in seen and code(9, 1, 8) in seen
    assert code(4, 1, 8) in seen and code(4, 1, 16) in seen
    assert not seen & UNREACHABLE


def test_every_reachable_kernel_was_compared():
    """Runs last: the flavour tests above launched exactly the reachable kernels, each compared with the oracle."""
    if len(DONE) < len(FLAVOURS) * len(VARIANTS):
        pytest.skip("needs every test_flavour case of this session to have passed")
    assert SEEN == REACHABLE, "missing %s, unexpected %s" % (
        sorted(hex(x) for x in REACHABLE - SEEN), sorted(hex(x) for x in SEEN - REACHABLE))
