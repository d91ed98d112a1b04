"""CPU tests of the 16-bit result entries (sm_*16, sm_download_web_u16): declared, exported, bound, and every one
rejects a NULL handle and bad arguments before it touches a device.  The handle-free checks come first in each
entry, so a dummy handle that is never dereferenced stands in for a context here; the checks that need a real
context (strides, band contexts) are in test_gpu_web16.py."""
import ctypes as C

import pytest

import stereomatching_b200 as smb

NEW = ["sm_match_wta_dev_batch16", "sm_run_batch16", "sm_multi_run_batch16", "sm_bands_run16", "sm_download_web_u16"]


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
    _fails(L.sm_match_wta_dev_batch16(None, 1, q, q, 16, p, p, 16), L, "NULL context")
    _fails(L.sm_run_batch16(None, 1, q, q, 0.15, p, p), L, "NULL context")
    _fails(L.sm_download_web_u16(None, p), L, "NULL context")
    _fails(L.sm_multi_run_batch16(None, 1, q, q, 0.15, p, p), L, "bad arguments")
    _fails(L.sm_bands_run16(None, q, q, 0.15, p, p), L, "bad arguments")


def test_bad_arguments_before_the_device(L, dummy):
    _, h = dummy
    buf = (C.c_uint16 * 16)()
    img = (C.c_uint8 * 16)()
    p, q = C.cast(buf, C.c_void_p), C.cast(img, C.c_void_p)
    # sm_match_wta_dev_batch16: NULL web, NULL edge maps, negative pair count (best may be NULL)
    _fails(L.sm_match_wta_dev_batch16(h, 1, q, q, 16, p, None, 16), L, "sm_match_wta_dev_batch16: bad arguments")
    _fails(L.sm_match_wta_dev_batch16(h, 1, None, q, 16, p, p, 16), L, "sm_match_wta_dev_batch16: bad arguments")
    _fails(L.sm_match_wta_dev_batch16(h, 1, q, None, 16, None, p, 16), L, "sm_match_wta_dev_batch16: bad arguments")
    _fails(L.sm_match_wta_dev_batch16(h, -1, q, q, 16, p, p, 16), L, "sm_match_wta_dev_batch16: bad arguments")
    # sm_run_batch16: NULL web / images, negative pair count, threshold out of [0, 1]
    _fails(L.sm_run_batch16(h, 1, q, q, 0.15, None, p), L, "sm_run_batch16: bad arguments")
    _fails(L.sm_run_batch16(h, 1, None, q, 0.15, p, p), L, "sm_run_batch16: bad arguments")
    _fails(L.sm_run_batch16(h, -2, q, q, 0.15, p, None), L, "sm_run_batch16: bad arguments")
    _fails(L.sm_run_batch16(h, 1, q, q, 1.5, p, None), L, "sm_run_batch16: threshold")
    _fails(L.sm_run_batch16(h, 1, q, q, -0.1, p, None), L, "sm_run_batch16: threshold")
    # sm_multi_run_batch16 / sm_bands_run16: NULL web / images, negative pair count
    _fails(L.sm_multi_run_batch16(h, 1, q, q, 0.15, None, p), L, "sm_multi_run_batch16: bad arguments")
    _fails(L.sm_multi_run_batch16(h, 1, q, None, 0.15, p, p), L, "sm_multi_run_batch16: bad arguments")
    _fails(L.sm_multi_run_batch16(h, -1, q, q, 0.15, p, None), L, "sm_multi_run_batch16: bad arguments")
    _fails(L.sm_bands_run16(h, q, q, 0.15, None, p), L, "sm_bands_run16: bad arguments")
    _fails(L.sm_bands_run16(h, None, q, 0.15, p, None), L, "sm_bands_run16: bad arguments")
    # sm_download_web_u16: NULL host array
    _fails(L.sm_download_web_u16(h, None), L, "sm_download_web_u16: NULL host pointer")


def test_binding_rejects_web16_with_web_u8():
    import numpy as np
    ctx = smb.StereoContext.__new__(smb.StereoContext)  # no device: the check comes before any call
    ctx.W, ctx.H, ctx._c = 8, 4, C.c_void_p()
    z = np.zeros((1, 4, 8), np.uint8)
    with pytest.raises(ValueError):
        ctx.run_batch(z, z, web_u8=True, web16=True)
