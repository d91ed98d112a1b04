"""CPU tests of the search-range creators (sm_create_range, sm_create_band_range, sm_multi_create_range,
sm_bands_create_range): declared, exported, bound, and every one rejects a bad range -- and the checks the creators
it extends already made -- with SM_ERR_ARG before it touches a device.  The Python keywords reach them."""
import ctypes as C

import pytest

import stereomatching_b200 as smb

NEW = ["sm_create_range", "sm_create_band_range", "sm_multi_create_range", "sm_bands_create_range"]


@pytest.fixture(scope="module")
def L():
    return smb.lib()


def _fails(rc, L, what):
    assert rc == -1, rc
    assert what.encode() in L.sm_last_error(), L.sm_last_error()


def _range_accepted(rc, L):
    """The range checks passed: whatever happens next (no device here) is not a rejection of the range."""
    assert not (rc == -1 and b"min_shift" in L.sm_last_error()), L.sm_last_error()


def test_entries_are_declared_bound_and_exported(L):
    for name in NEW:
        assert name in smb.SYMBOLS
        assert getattr(L, name).argtypes is not None, name


def test_abi_version_stays_1_3(L):
    assert L.sm_version() == (1 << 16) | 3


def _creators(L):
    """Each creator as f(min_shift, num_shifts, **overrides) -> status, on a 64 x 64 frame, window 9, WRAP."""
    devs = (C.c_int * 2)(0, 0)

    def ctx(m, d, w=64, h=64, sw=9, v=0):
        p = C.c_void_p()
        return L.sm_create_range(C.byref(p), 0, w, h, m, d, sw, v)

    def band(m, d, w=64, h=64, sw=9, v=0, r0=8, r1=40):
        p = C.c_void_p()
        return L.sm_create_band_range(C.byref(p), 0, w, h, r0, r1, m, d, sw, v)

    def multi(m, d, w=64, h=64, sw=9, v=0, n=2):
        p = C.c_void_p()
        return L.sm_multi_create_range(C.byref(p), devs, n, w, h, m, d, sw, v)

    def bands(m, d, w=64, h=64, sw=9, v=0, n=2):
        p = C.c_void_p()
        return L.sm_bands_create_range(C.byref(p), devs, n, w, h, m, d, sw, v)

    return {"sm_create_range": ctx, "sm_create_band_range": band, "sm_multi_create_range": multi,
            "sm_bands_create_range": bands}


@pytest.mark.parametrize("name", NEW)
def test_range_is_checked_before_the_device(L, name):
    f = _creators(L)[name]
    _fails(f(-1, 30), L, "min_shift")
    _fails(f(-(1 << 30), 1), L, "min_shift")
    _fails(f(65535 - 29, 30), L, "min_shift")       # web would reach 65536
    _fails(f(65535, 1), L, "min_shift")
    _fails(f((1 << 31) - 1, 512), L, "min_shift")   # no overflow in the check
    _range_accepted(f(65535 - 30, 30), L)          # the top of the range: min_shift + num_shifts == 65535
    _range_accepted(f(65535 - 512, 512), L)
    _range_accepted(f(0, 30), L)


@pytest.mark.parametrize("name", NEW)
def test_existing_checks_stay(L, name):
    f = _creators(L)[name]
    _fails(f(5, 0), L, "num_shifts")
    _fails(f(5, 513), L, "num_shifts")
    _fails(f(5, 30, w=0), L, "width/height")
    _fails(f(5, 30, sw=64), L, "square_width")
    _fails(f(5, 30, w=20, sw=21), L, "square width")
    _fails(f(5, 30, v=2), L, "variant")


def test_creator_specific_checks(L):
    p = C.c_void_p()
    devs = (C.c_int * 2)(0, 0)
    _fails(L.sm_create_range(None, 0, 64, 64, 5, 30, 9, 0), L, "NULL ctx")
    _fails(L.sm_create_band_range(C.byref(p), 0, 64, 64, 10, 5, 5, 30, 9, 0), L, "bad row band")
    _fails(L.sm_create_band_range(C.byref(p), 0, 64, 64, 0, 65, 5, 30, 9, 0), L, "bad row band")
    _fails(L.sm_multi_create_range(C.byref(p), None, 2, 64, 64, 5, 30, 9, 0), L, "sm_multi_create: bad arguments")
    _fails(L.sm_multi_create_range(C.byref(p), devs, 0, 64, 64, 5, 30, 9, 0), L, "sm_multi_create: bad arguments")
    _fails(L.sm_bands_create_range(C.byref(p), devs, 0, 64, 64, 5, 30, 9, 0), L, "sm_bands_create: bad arguments")
    _fails(L.sm_bands_create_range(C.byref(p), devs, 2, 64, 1, 5, 30, 1, 0), L, "fewer rows than bands")


def test_old_creators_are_the_zero_range(L):
    """The creators without a range reject exactly what their range twin rejects at min_shift 0."""
    p = C.c_void_p()
    devs = (C.c_int * 1)(0)
    _fails(L.sm_create(C.byref(p), 0, 64, 64, 513, 9, 0), L, "num_shifts")
    _range_accepted(L.sm_create(C.byref(p), 0, 64, 64, 512, 9, 0), L)
    _fails(L.sm_create_band(C.byref(p), 0, 64, 64, 0, 64, 0, 9, 0), L, "num_shifts")
    _fails(L.sm_multi_create(C.byref(p), devs, 1, 64, 64, 0, 9, 0), L, "num_shifts")
    _fails(L.sm_bands_create(C.byref(p), devs, 1, 64, 64, 0, 9, 0), L, "num_shifts")


@pytest.mark.parametrize("make", [
    lambda m, d: smb.StereoContext(64, 64, d, 9, smb.WRAP, min_shift=m),
    lambda m, d: smb.StereoContext(64, 64, d, 9, smb.GHOST, rows=(8, 40), min_shift=m),
    lambda m, d: smb.MultiGpuBatch([0, 0], 64, 64, d, 9, min_shift=m),
    lambda m, d: smb.MultiGpuBands([0, 0], 64, 64, d, 9, min_shift=m),
], ids=["StereoContext", "StereoContext_band", "MultiGpuBatch", "MultiGpuBands"])
def test_python_keyword_reaches_the_creator(make):
    for m, d in ((-1, 30), (65535 - 29, 30), (65535, 1)):
        with pytest.raises(smb.StereoError) as e:
            make(m, d)
        assert e.value.code == -1 and "min_shift" in str(e.value), e.value
    # an accepted range fails (here, without a device) only after the range checks
    try:
        make(65535 - 30, 30).close()
    except smb.StereoError as e:
        assert "min_shift" not in str(e), e
