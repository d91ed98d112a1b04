"""CPU tests of the entries with both extras (sm_*_ru_sub16): declared, exported, bound, and every one rejects a NULL
handle, a NULL runner_up / web_sub / web array, NULL inputs, a negative pair count and a threshold outside [0, 1]
before it touches a device.  The handle-free checks come first in each entry, so a dummy handle that is never
dereferenced stands in for a context here."""
import ctypes as C

import numpy as np
import pytest

import stereomatching_b200 as smb

NEW = ["sm_match_wta_dev_batch_ru_sub16", "sm_run_batch_ru_sub16", "sm_multi_run_batch_ru_sub16",
       "sm_bands_run_ru_sub16"]


@pytest.fixture(scope="module")
def L():
    return smb.lib()


@pytest.fixture(scope="module")
def dummy():
    """A non-NULL handle the argument checks under test never dereference."""
    buf = C.create_string_buffer(4096)
    return buf, C.c_void_p(C.addressof(buf))


def _fails(rc, L, what):
    assert rc == -1, rc
    assert what.encode() in L.sm_last_error(), L.sm_last_error()


def test_entries_are_declared_bound_and_exported(L):
    for name in NEW:
        assert name in smb.SYMBOLS
        assert getattr(L, name).argtypes is not None, name


def test_abi_version_stays_1_3(L):
    assert L.sm_version() == (1 << 16) | 3


def test_null_handles(L):
    buf = (C.c_uint16 * 16)()
    img = (C.c_uint8 * 16)()
    p, q = C.cast(buf, C.c_void_p), C.cast(img, C.c_void_p)
    _fails(L.sm_match_wta_dev_batch_ru_sub16(None, 1, q, q, 16, p, p, p, p, 16), L, "NULL context")
    _fails(L.sm_run_batch_ru_sub16(None, 1, q, q, 0.15, p, p, p, p), L, "NULL context")
    _fails(L.sm_multi_run_batch_ru_sub16(None, 1, q, q, 0.15, p, p, p, p), L, "bad arguments")
    _fails(L.sm_bands_run_ru_sub16(None, q, q, 0.15, p, p, p, p), L, "bad arguments")


def test_bad_arguments_before_the_device(L, dummy):
    _, h = dummy
    buf = (C.c_uint16 * 16)()
    img = (C.c_uint8 * 16)()
    p, q = C.cast(buf, C.c_void_p), C.cast(img, C.c_void_p)
    f = "sm_match_wta_dev_batch_ru_sub16: bad arguments"
    fn = L.sm_match_wta_dev_batch_ru_sub16
    _fails(fn(h, 1, q, q, 16, p, p, None, p, 16), L, f)  # NULL runner_up
    _fails(fn(h, 1, q, q, 16, p, p, p, None, 16), L, f)  # NULL web_sub
    _fails(fn(h, 1, q, q, 16, p, None, p, p, 16), L, f)  # NULL web
    _fails(fn(h, 1, None, q, 16, p, p, p, p, 16), L, f)
    _fails(fn(h, 1, q, None, 16, None, p, p, p, 16), L, f)
    _fails(fn(h, -1, q, q, 16, p, p, p, p, 16), L, f)
    for name in ("sm_run_batch_ru_sub16", "sm_multi_run_batch_ru_sub16"):
        fn = getattr(L, name)
        bad = name + ": bad arguments"
        _fails(fn(h, 1, q, q, 0.15, p, p, None, p), L, bad)  # NULL runner_up (best may be NULL)
        _fails(fn(h, 1, q, q, 0.15, p, None, p, None), L, bad)  # NULL web_sub
        _fails(fn(h, 1, q, q, 0.15, None, p, p, p), L, bad)
        _fails(fn(h, 1, None, q, 0.15, p, p, p, p), L, bad)
        _fails(fn(h, 1, q, None, 0.15, p, None, p, p), L, bad)
        _fails(fn(h, -2, q, q, 0.15, p, None, p, p), L, bad)
        _fails(fn(h, 1, q, q, 1.5, p, None, p, p), L, name + ": threshold")
        _fails(fn(h, 1, q, q, -0.1, p, None, p, p), L, name + ": threshold")
    fn, bad = L.sm_bands_run_ru_sub16, "sm_bands_run_ru_sub16: bad arguments"
    _fails(fn(h, q, q, 0.15, p, p, None, p), L, bad)
    _fails(fn(h, q, q, 0.15, p, p, p, None), L, bad)
    _fails(fn(h, q, q, 0.15, None, p, p, p), L, bad)
    _fails(fn(h, None, q, 0.15, p, None, p, p), L, bad)
    _fails(fn(h, q, q, 2.0, p, None, p, p), L, "sm_bands_run_ru_sub16: threshold")
    _fails(fn(h, q, q, -1.0, p, None, p, p), L, "sm_bands_run_ru_sub16: threshold")


def _unbound():
    """The three Python classes with NULL handles: nothing reaches a device."""
    ctx = smb.StereoContext.__new__(smb.StereoContext)
    ctx.W, ctx.H, ctx._c = 8, 4, C.c_void_p()
    multi = smb.MultiGpuBatch.__new__(smb.MultiGpuBatch)
    multi.W, multi.H, multi._m = 8, 4, C.c_void_p()
    bands = smb.MultiGpuBands.__new__(smb.MultiGpuBands)
    bands.W, bands.H, bands._b = 8, 4, C.c_void_p()
    return ctx, multi, bands


@pytest.mark.parametrize("threshold", [-0.1, 1.5])
def test_binding_rejects_what_the_siblings_reject(threshold):
    """A threshold outside [0, 1], a NULL handle and a wrongly shaped input fail in the combined methods as in
    run_batch(web16=True, want_runner_up=True) / want_subpixel=True and in bands.run."""
    ctx, multi, bands = _unbound()
    z = np.zeros((1, 4, 8), np.uint8)
    for obj, both, sibling in ((ctx, ctx.run_batch_ru_sub16, ctx.run_batch),
                               (multi, multi.run_batch_ru_sub16, multi.run_batch)):
        for kw in ({"want_runner_up": True}, {"want_subpixel": True}):
            with pytest.raises(smb.StereoError) as sib:
                sibling(z, z, threshold, web16=True, **kw)
            with pytest.raises(smb.StereoError) as got:
                both(z, z, threshold)
            assert ("threshold" in str(sib.value)) == ("threshold" in str(got.value)), (str(sib.value), str(got.value))
        with pytest.raises(smb.StereoError):
            both(z, z, 0.15, want_best=True)  # the NULL handle
        with pytest.raises(AssertionError):
            both(np.zeros((1, 4, 9), np.uint8), z)
    for kw in ({"want_runner_up": True}, {"want_subpixel": True}):
        with pytest.raises(smb.StereoError):
            bands.run(z[0], z[0], threshold, web16=True, **kw)
    for t in (threshold, 0.15):  # (the NULL handle fails first, as in the siblings)
        with pytest.raises(smb.StereoError, match="sm_bands_run_ru_sub16: bad arguments"):
            bands.run_ru_sub16(z[0], z[0], t)
    with pytest.raises(AssertionError):
        bands.run_ru_sub16(z[0, :, :7], z[0])


def test_run_batch_flags_stay_exclusive():
    """Both extras come from the *_ru_sub16 methods; the flags of run_batch / run keep excluding each other."""
    ctx, multi, bands = _unbound()
    z = np.zeros((1, 4, 8), np.uint8)
    with pytest.raises(ValueError, match="ru_sub16"):
        ctx.run_batch(z, z, web16=True, want_subpixel=True, want_runner_up=True)
    with pytest.raises(ValueError, match="ru_sub16"):
        multi.run_batch(z, z, web16=True, want_subpixel=True, want_runner_up=True)
    with pytest.raises(ValueError, match="ru_sub16"):
        bands.run(z[0], z[0], web16=True, want_subpixel=True, want_runner_up=True)
