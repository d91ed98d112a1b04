"""The 16-bit result entries on the GPU: sm_match_wta_dev_batch16 (the k_bitslice16 / k_direct16 kernels),
sm_run_batch16, sm_multi_run_batch16, sm_bands_run16, sm_download_web_u16 and `stereobatch ... u16`.

Every reachable instantiation of the 16-bit bit-sliced family is compared with the oracle and with the int32 entry
on the same inputs (the flavour table of test_gpu_flavours.py), in one-pair and several-pairs launches, with and
without a best array, and reports the shape code of the int32 kernel it mirrors.  Outputs sit in buffers whose pairs
are further apart than a frame, with guard elements of 0xFFFF that must survive every launch.  The BASELINE configs
3 and 4 go through the host-buffer entries against the reference's CRCs (golden.json)."""
import os
import subprocess
import zlib

import numpy as np
import pytest

import oracle
import stereomatching_b200 as smb
from test_gpu_flavours import FLAVOURS, REACHABLE, code, expected_shape, families, reference, run_dev_batch
from util import ROOT, THRESHOLD, vname

pytestmark = pytest.mark.gpu

VARIANTS = [smb.WRAP, smb.GHOST]
GUARD = 37      # elements between one pair's frame and the next one's
SEEN16 = set()  # shape codes of the 16-bit launches compared with the oracle by test_flavour16
DONE16 = set()


@pytest.fixture(scope="module")
def num_sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def run16(c, les, res, with_best=True, rows=None):
    """sm_match_wta_dev_batch16 over distinct pairs, outputs out_stride = H*W + GUARD apart in buffers filled with
    0xFFFF.  Asserts that nothing outside the frames (and, for a band context, outside its rows [r0, r1)) was
    written; returns (best, web) as (n, H, W) int32 arrays (best None without)."""
    import torch
    n, (H, W) = len(les), les[0].shape
    npix, stride = H * W, H * W + GUARD
    d1 = torch.from_numpy(np.stack(les)).cuda()
    d2 = torch.from_numpy(np.stack(res)).cuda()
    web = torch.full((n * stride + GUARD,), -1, dtype=torch.int16, device="cuda")  # 0xFFFF
    best = torch.full((n * stride + GUARD,), -1, dtype=torch.int16, device="cuda") if with_best else None
    torch.cuda.synchronize()
    c.match_wta_dev_batch16(n, d1.data_ptr(), d2.data_ptr(), npix, best.data_ptr() if with_best else None,
                            web.data_ptr(), stride)
    c.synchronize()
    out = []
    for buf in (best, web):
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
    return out[0], out[1]


def at(a, k):
    return None if a is None else a[k]


def check(best, web, bo, wo, what):
    if best is not None:
        assert np.array_equal(best, bo), "%s: best differs in %d pixels" % (what, (best != bo).sum())
    assert np.array_equal(web, wo), "%s: web differs in %d pixels" % (what, (web != wo).sum())


# ---------------------------------------------------------------------------------
# every reachable k_bitslice16 instantiation
# ---------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
@pytest.mark.parametrize("flavour", list(FLAVOURS))
def test_flavour16(orc, num_sms, flavour, variant):
    nw, seg, multi, c2, hp, halves, geometry = FLAVOURS[flavour]
    for half in halves:
        want = code(half, nw, seg, c2, hp, multi)
        W, H1, Hn, D = geometry(half, num_sms)
        sw = 2 * half + 1
        seed = 7000 + 1000 * half + 17 * D + W
        tag = "%s half %d %dx%d D %d %s" % (flavour, half, W, H1, D, vname(variant))
        fams = families(W, H1, D, seed)
        refs = {name: reference(orc, name, le, re, D, sw, variant) for name, le, re in fams}
        with smb.StereoContext(W, H1, D, sw, variant, kernel=smb.KERNEL_BITSLICE) as c:
            # the int32 entry's one-pair launch on the first input: the 16-bit one must report its shape
            b32, w32 = run_dev_batch(c, [fams[0][1]], [fams[0][2]])
            shape32 = c.get_info(smb.INFO_KERNEL_SHAPE)
            assert shape32 == want, tag
            for k, (name, le, re) in enumerate(fams):
                for with_best in (True, False) if k < 2 else (True,):
                    best, web = run16(c, [le], [re], with_best)
                    what = "%s %s one pair%s" % (tag, name, "" if with_best else ", no best")
                    assert c.get_info(smb.INFO_KERNEL_SHAPE) == shape32, what
                    SEEN16.add(c.get_info(smb.INFO_KERNEL_SHAPE))
                    check(at(best, 0), web[0], *refs[name], what)
                    if k == 0:
                        check(at(best, 0), web[0], b32[0], w32[0], what + " vs int32")
        if Hn is not None:
            if Hn != H1:
                fams = families(W, Hn, D, seed + 1)
                refs = {name: reference(orc, name, le, re, D, sw, variant) for name, le, re in fams}
            with smb.StereoContext(W, Hn, D, sw, variant, kernel=smb.KERNEL_BITSLICE) as c:
                les, res = [f[1] for f in fams], [f[2] for f in fams]
                b32, w32 = run_dev_batch(c, les, res)
                shape32 = c.get_info(smb.INFO_KERNEL_SHAPE)
                for with_best in (True, False):
                    best, web = run16(c, les, res, with_best)
                    what = "%s, %d pairs per call%s" % (tag, len(fams), "" if with_best else ", no best")
                    assert c.get_info(smb.INFO_KERNEL_SHAPE) == shape32 == want, what
                    SEEN16.add(want)
                    for k, (name, _, _) in enumerate(fams):
                        check(at(best, k), web[k], *refs[name], "%s, pair %d (%s)" % (what, k, name))
                        check(at(best, k), web[k], b32[k], w32[k], "%s, pair %d vs int32" % (what, k))
        # a band context: rows [r0, r1) only, the others keep their guard value
        name, le, re = fams[1] if Hn is None or Hn == H1 else families(W, H1, D, seed)[1]
        bo, wo = reference(orc, name, le, re, D, sw, variant)
        r0, r1 = H1 // 3, H1 // 3 + max(1, min(H1 // 3, 20))
        with smb.StereoContext(W, H1, D, sw, variant, rows=(r0, r1), kernel=smb.KERNEL_BITSLICE) as c:
            best, web = run16(c, [le], [re], True, rows=(r0, r1))
            assert c.get_info(smb.INFO_KERNEL_SHAPE) == expected_shape(W, r1 - r0, D, half, 1, num_sms)
        check(best[0, r0:r1], web[0, r0:r1], bo[r0:r1], wo[r0:r1], "%s band [%d, %d)" % (tag, r0, r1))
    DONE16.add((flavour, variant))


@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
def test_odd_widths_and_selection_switches(orc, num_sms, variant):
    """Frames on both sides of the selection switches, odd widths among them: the 16-bit launch picks the int32
    launch's kernel and writes nothing past a row's last pixel."""
    cases = [(w, 40, 30, h) for h in (2, 6, 7) for w in (63, 65)]
    cases += [(w, 40, 16, h) for h in (3, 9) for w in (63, 65, 127, 129)]
    cases += [(97, 41, 70, 4), (33, 23, 200, 1)]
    for W, H, D, half in cases:
        sw = 2 * half + 1
        rng = np.random.default_rng(W * 1000 + H + half)
        les = [(rng.random((H, W)) < d).astype(np.uint8) for d in (0.2, 0.6)]
        res = [np.roll(le, k + 3, axis=1) ^ (rng.random((H, W)) < 0.03).astype(np.uint8) for k, le in enumerate(les)]
        refs = [reference(orc, "random", le, re, D, sw, variant) for le, re in zip(les, res)]
        tag = "%dx%d D %d half %d" % (W, H, D, half)
        with smb.StereoContext(W, H, D, sw, variant) as c:
            for n in (1, 2):
                best, web = run16(c, les[:n], res[:n])
                assert c.get_info(smb.INFO_KERNEL_SHAPE) == expected_shape(W, H, D, half, n, num_sms), tag
                for k in range(n):
                    check(best[k], web[k], *refs[k], "%s, %d pairs, pair %d" % (tag, n, k))


# ---------------------------------------------------------------------------------
# more than 64 shifts: the chunks merge through a u16 best
# ---------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
@pytest.mark.parametrize("D", [65, 129, 256, 512])
def test_multi_chunks(orc, variant, D):
    W, H, sw = 128, 24, 9
    fams = [f for f in families(W, H, D, 31 * D + variant) if f[0].startswith("periodic") or f[0] == "random0.60"]
    assert len(fams) == 4
    refs = {name: reference(orc, name, le, re, D, sw, variant) for name, le, re in fams}
    with smb.StereoContext(W, H, D, sw, variant) as c:
        for with_best in (True, False):
            for name, le, re in fams:  # one pair per launch
                best, web = run16(c, [le], [re], with_best)
                assert c.get_info(smb.INFO_KERNEL_SHAPE) & smb.SHAPE_MULTI
                check(at(best, 0), web[0], *refs[name], "D %d %s one pair, best %s" % (D, name, with_best))
            best, web = run16(c, [f[1] for f in fams], [f[2] for f in fams], with_best)
            for k, (name, _, _) in enumerate(fams):
                check(at(best, k), web[k], *refs[name], "D %d %s in a batch, best %s" % (D, name, with_best))


@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
@pytest.mark.parametrize("W,H,D,sw", [(48, 40, 30, 21), (64, 40, 129, 9)], ids=["one_word", "chunks"])
def test_ragged_batch(orc, variant, W, H, D, sw):
    """17 pairs: a launch of 16, then one of a single pair (the one-pair shape; the 8-pixel-segment kernel for the
    small one-word frame), with and without best; the last launch's shape is the int32 entry's."""
    n = 17
    rng = np.random.default_rng(170 + D + variant)
    les = [(rng.random((H, W)) < (0.1 + 0.04 * k)).astype(np.uint8) for k in range(n)]
    res = [np.roll(le, k % D, axis=1) ^ (rng.random((H, W)) < 0.02).astype(np.uint8) for k, le in enumerate(les)]
    with smb.StereoContext(W, H, D, sw, variant) as c:
        b32, w32 = run_dev_batch(c, les, res)
        shape32 = c.get_info(smb.INFO_KERNEL_SHAPE)
        assert c.get_info(smb.INFO_PAIRS_PER_LAUNCH) == 16
        for with_best in (True, False):
            best, web = run16(c, les, res, with_best)
            assert c.get_info(smb.INFO_KERNEL_SHAPE) == shape32
            assert c.last_launches() == 4  # two groups: a pack and a main kernel each
            for k in range(n):
                check(at(best, k), web[k], b32[k], w32[k], "pair %d, best %s" % (k, with_best))
    for k in (0, 15, 16):
        check(None, w32[k], *reference(orc, "random", les[k], res[k], D, sw, variant), "int32 pair %d" % k)
    if sw == 21:
        assert shape32 == code(10, 1, 8)


# ---------------------------------------------------------------------------------
# the direct kernel's 16-bit twin
# ---------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
@pytest.mark.parametrize("sw", [33, 45, 63])
def test_direct_wide_windows(orc, variant, sw):
    W, H, D = 70, 66, 20
    name, le, re = families(W, H, D, sw + variant)[1]
    bo, wo = reference(orc, name, le, re, D, sw, variant)
    with smb.StereoContext(W, H, D, sw, variant) as c:
        for with_best in (True, False):
            best, web = run16(c, [le, le], [re, re], with_best)
            assert c.get_info(smb.INFO_KERNEL_SHAPE) == smb.SHAPE_DIRECT
            for k in range(2):
                check(at(best, k), web[k], bo, wo, "window %d, best %s" % (sw, with_best))


@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
def test_direct_forced(orc, variant):
    W, H, D, sw = 64, 40, 50, 9
    fams = families(W, H, D, 50 + variant)
    with smb.StereoContext(W, H, D, sw, variant, kernel=smb.KERNEL_DIRECT) as c:
        les, res = [f[1] for f in fams], [f[2] for f in fams]
        for with_best in (True, False):
            best, web = run16(c, les, res, with_best)
            assert c.get_info(smb.INFO_KERNEL_SHAPE) == smb.SHAPE_DIRECT
            for k, (name, le, re) in enumerate(fams):
                check(at(best, k), web[k], *reference(orc, name, le, re, D, sw, variant), name)


# ---------------------------------------------------------------------------------
# arguments that need a context
# ---------------------------------------------------------------------------------
def test_arguments_with_a_context():
    import torch
    W, H = 64, 32
    L = smb.lib()
    e = torch.zeros((2, H, W), dtype=torch.uint8, device="cuda")
    o = torch.zeros((2, H * W), dtype=torch.int16, device="cuda")
    with smb.StereoContext(W, H, 40, 9) as c:
        with pytest.raises(smb.StereoError, match="stride below frame size"):
            c.match_wta_dev_batch16(1, e.data_ptr(), e.data_ptr(), H * W - 1, None, o.data_ptr(), H * W)
        with pytest.raises(smb.StereoError, match="stride below frame size"):
            c.match_wta_dev_batch16(1, e.data_ptr(), e.data_ptr(), H * W, None, o.data_ptr(), H * W - 1)
        c.match_wta_dev_batch16(0, e.data_ptr(), e.data_ptr(), H * W, None, o.data_ptr(), H * W)  # nothing to do
        with pytest.raises(smb.StereoError, match="no web"):
            c.download_web_u16()
    with smb.StereoContext(W, H, 40, 9, rows=(4, 20)) as c:
        z = np.zeros((1, H, W), np.uint8)
        with pytest.raises(smb.StereoError, match="whole-frame contexts only"):
            c.run_batch(z, z, web16=True)
        assert L.sm_run_batch16(c._c, 1, z.ctypes.data, z.ctypes.data, 0.15, None, None) == -1


# ---------------------------------------------------------------------------------
# host-buffer entries against the reference's CRCs
# ---------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
def test_config3_bands16(orc, golden, variant):
    """Config 3 (3840x2160, 256 shifts, window 11) through sm_bands_run16, every slot on device 0: 1, 2 and 8
    bands, with and without best; the frame is filled with 0xFFFF first, so every row must have been written."""
    g = golden["synth/c3/%s" % vname(variant)]
    left, right, _ = orc.synth_pair(g["seed"], g["w"], g["h"], g["D"])
    for nb in (1, 2, 8):
        with smb.MultiGpuBands([0] * nb, g["w"], g["h"], g["D"], g["sw"], variant) as b:
            web, best = b.run(left, right, THRESHOLD, want_best=True, web16=True)
            assert web.dtype == best.dtype == np.uint16
            assert oracle.crc32(web.astype(np.int32)) == g["web"], nb
            assert oracle.crc32(best.astype(np.int32)) == g["best"], nb
            web_only = b.run(left, right, THRESHOLD, web16=True)
            assert np.array_equal(web_only, web), nb


@pytest.mark.parametrize("variant", VARIANTS, ids=vname)
def test_config4_batch16(orc, golden, variant):
    """Config 4 (1280x720, 128 shifts, window 21): the four reference-pinned pairs repeated to 10 through
    sm_run_batch16 and sm_multi_run_batch16 (slots [0, 0])."""
    gs = [golden["synth/c4/%d/%s" % (k, vname(variant))] for k in range(4)]
    pairs = [orc.synth_pair(g["seed"], g["w"], g["h"], g["D"]) for g in gs]
    n = 10
    first = np.stack([pairs[k % 4][0] for k in range(n)])
    second = np.stack([pairs[k % 4][1] for k in range(n)])
    g0 = gs[0]
    with smb.StereoContext(g0["w"], g0["h"], g0["D"], g0["sw"], variant) as c:
        web, best = c.run_batch(first, second, THRESHOLD, want_best=True, web16=True)
        web_only = c.run_batch(first, second, THRESHOLD, web16=True)
    with smb.MultiGpuBatch([0, 0], g0["w"], g0["h"], g0["D"], g0["sw"], variant) as m:
        mweb, mbest = m.run_batch(first, second, THRESHOLD, want_best=True, web16=True)
    for k in range(n):
        for w_, b_ in ((web, best), (mweb, mbest)):
            assert w_.dtype == b_.dtype == np.uint16
            assert oracle.crc32(w_[k].astype(np.int32)) == gs[k % 4]["web"], k
            assert oracle.crc32(b_[k].astype(np.int32)) == gs[k % 4]["best"], k
    assert np.array_equal(web_only, web)


@pytest.mark.parametrize("D", [30, 300, 512])
def test_download_web_u16(D):
    W, H, sw = 96, 40, 9
    rng = np.random.default_rng(D)
    le = (rng.random((H, W)) < 0.5).astype(np.uint8)
    re = np.roll(le, 5, axis=1) ^ (rng.random((H, W)) < 0.05).astype(np.uint8)
    with smb.StereoContext(W, H, D, sw) as c:
        _, web = c.match_wta_host(le, re)
        w16 = c.download_web_u16()
        assert w16.dtype == np.uint16 and np.array_equal(w16.astype(np.int32), web)
    with smb.StereoContext(W, H, D, sw, rows=(7, 23)) as c:  # a band context writes only its rows
        c.set_edges(le, re)
        c.match_wta()
        w16 = c.download_web_u16(out=np.full((H, W), 0xFFFF, np.uint16))
        assert np.array_equal(w16[7:23].astype(np.int32), web[7:23])
        assert (w16[:7] == 0xFFFF).all() and (w16[23:] == 0xFFFF).all()


def test_stereobatch_u16(orc):
    """`stereobatch ... u16` runs sm_multi_run_batch16; its web CRC equals that of the i32 run's webs as uint16."""
    exe = os.path.join(ROOT, "timing", "stereobatch")
    assert os.path.exists(exe), "run `make build=timing` (or __graft_entry__.build())"
    w, h, D, sw, n = 320, 180, 300, 9, 3
    webs = []
    for k in range(n):
        left, right, _ = orc.synth_pair(1234 + 2 * k, w, h, D)
        e1, e2 = orc.edges(left, THRESHOLD, 0), orc.edges(right, THRESHOLD, 0)
        webs.append(orc.match_wta(e1, e2, D, sw, 0)[1])
    webs = np.stack(webs)
    for kind, dt in (("i32", np.int32), ("u16", np.uint16)):
        r = subprocess.run([exe, str(w), str(h), str(D), str(sw), str(n), "wrap", kind], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        fields = dict(kv.split(" = ") for kv in r.stdout.strip().split(", "))
        assert fields["web_crc32"] == "%08x" % (zlib.crc32(webs.astype(dt).tobytes()) & 0xFFFFFFFF), (kind, r.stdout)


def test_every_reachable_kernel_ran_in_16_bits():
    """Runs last: test_flavour16 launched exactly the reachable set of k_bitslice16 instantiations."""
    if len(DONE16) < len(FLAVOURS) * len(VARIANTS):
        pytest.skip("needs every test_flavour16 case of this session to have passed")
    assert SEEN16 == REACHABLE, "missing %s, unexpected %s" % (
        sorted(hex(x) for x in REACHABLE - SEEN16), sorted(hex(x) for x in SEEN16 - REACHABLE))
