"""CPU tests of the sub-pixel entries (sm_*_sub16): declared, exported, bound, and every one rejects a NULL handle,
a NULL web_sub array, NULL inputs and a threshold outside [0, 1] before it touches a device.  The handle-free
checks come first in each entry, so a dummy handle that is never dereferenced stands in for a context here."""
import ctypes as C

import numpy as np
import pytest

import stereomatching_b200 as smb

NEW = ["sm_match_wta_dev_batch_sub16", "sm_run_batch_sub16", "sm_multi_run_batch_sub16", "sm_bands_run_sub16"]


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
    _fails(L.sm_match_wta_dev_batch_sub16(None, 1, q, q, 16, p, p, p, 16), L, "NULL context")
    _fails(L.sm_run_batch_sub16(None, 1, q, q, 0.15, p, p, p), L, "NULL context")
    _fails(L.sm_multi_run_batch_sub16(None, 1, q, q, 0.15, p, p, p), L, "bad arguments")
    _fails(L.sm_bands_run_sub16(None, q, q, 0.15, p, p, p), L, "bad arguments")


def test_bad_arguments_before_the_device(L, dummy):
    _, h = dummy
    buf = (C.c_uint16 * 16)()
    img = (C.c_uint8 * 16)()
    p, q = C.cast(buf, C.c_void_p), C.cast(img, C.c_void_p)
    f = "sm_match_wta_dev_batch_sub16: bad arguments"
    _fails(L.sm_match_wta_dev_batch_sub16(h, 1, q, q, 16, p, p, None, 16), L, f)  # NULL web_sub
    _fails(L.sm_match_wta_dev_batch_sub16(h, 1, q, q, 16, p, None, p, 16), L, f)  # NULL web
    _fails(L.sm_match_wta_dev_batch_sub16(h, 1, None, q, 16, p, p, p, 16), L, f)
    _fails(L.sm_match_wta_dev_batch_sub16(h, 1, q, None, 16, None, p, p, 16), L, f)
    _fails(L.sm_match_wta_dev_batch_sub16(h, -1, q, q, 16, p, p, p, 16), L, f)
    for name in ("sm_run_batch_sub16", "sm_multi_run_batch_sub16"):
        fn = getattr(L, name)
        _fails(fn(h, 1, q, q, 0.15, p, p, None), L, name + ": bad arguments")  # NULL web_sub (best may be NULL)
        _fails(fn(h, 1, q, q, 0.15, p, None, None), L, name + ": bad arguments")
        _fails(fn(h, 1, q, q, 0.15, None, p, p), L, name + ": bad arguments")
        _fails(fn(h, 1, None, q, 0.15, p, p, p), L, name + ": bad arguments")
        _fails(fn(h, 1, q, None, 0.15, p, None, p), L, name + ": bad arguments")
        _fails(fn(h, -2, q, q, 0.15, p, None, p), L, name + ": bad arguments")
        _fails(fn(h, 1, q, q, 1.5, p, None, p), L, name + ": threshold")
        _fails(fn(h, 1, q, q, -0.1, p, None, p), L, name + ": threshold")
    _fails(L.sm_bands_run_sub16(h, q, q, 0.15, p, p, None), L, "sm_bands_run_sub16: bad arguments")
    _fails(L.sm_bands_run_sub16(h, q, q, 0.15, None, p, p), L, "sm_bands_run_sub16: bad arguments")
    _fails(L.sm_bands_run_sub16(h, None, q, 0.15, p, None, p), L, "sm_bands_run_sub16: bad arguments")
    _fails(L.sm_bands_run_sub16(h, q, q, 2.0, p, None, p), L, "sm_bands_run_sub16: threshold")
    _fails(L.sm_bands_run_sub16(h, q, q, -1.0, p, None, p), L, "sm_bands_run_sub16: threshold")


def test_binding_needs_web16_for_web_sub():
    ctx = smb.StereoContext.__new__(smb.StereoContext)  # no device: the check comes before any call
    ctx.W, ctx.H, ctx._c = 8, 4, C.c_void_p()
    z = np.zeros((1, 4, 8), np.uint8)
    with pytest.raises(ValueError):
        ctx.run_batch(z, z, want_subpixel=True)
    bands = smb.MultiGpuBands.__new__(smb.MultiGpuBands)
    bands.W, bands.H, bands._b = 8, 4, C.c_void_p()
    with pytest.raises(ValueError):
        bands.run(z[0], z[0], want_subpixel=True)
    multi = smb.MultiGpuBatch.__new__(smb.MultiGpuBatch)
    multi.W, multi.H, multi._m = 8, 4, C.c_void_p()
    with pytest.raises(ValueError):
        multi.run_batch(z, z, want_subpixel=True)


def test_binding_rejects_web_sub_with_the_runner_up():
    ctx = smb.StereoContext.__new__(smb.StereoContext)
    ctx.W, ctx.H, ctx._c = 8, 4, C.c_void_p()
    z = np.zeros((1, 4, 8), np.uint8)
    with pytest.raises(ValueError):
        ctx.run_batch(z, z, web16=True, want_subpixel=True, want_runner_up=True)
    bands = smb.MultiGpuBands.__new__(smb.MultiGpuBands)
    bands.W, bands.H, bands._b = 8, 4, C.c_void_p()
    with pytest.raises(ValueError):
        bands.run(z[0], z[0], web16=True, want_subpixel=True, want_runner_up=True)
    multi = smb.MultiGpuBatch.__new__(smb.MultiGpuBatch)
    multi.W, multi.H, multi._m = 8, 4, C.c_void_p()
    with pytest.raises(ValueError):
        multi.run_batch(z, z, web16=True, want_subpixel=True, want_runner_up=True)
