"""ctypes binding of libstereo_b200.so (include/stereo_b200.h).

Thin by design: every method is one C-ABI call on host numpy buffers (or raw device
pointers for the ``*_dev`` calls).  There is NO fallback: if the shared library is
missing or a call fails, a ``StereoError`` is raised.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("STEREO_B200_LIB") or os.path.join(HERE, "libstereo_b200.so")

WRAP, GHOST = 0, 1
KERNEL_AUTO, KERNEL_DIRECT, KERNEL_BITSLICE = 0, 1, 2
OPT_EDGES_FP64, OPT_PIPE_GROUP, OPT_ROW_RUNS = 1, 2, 3
INFO_WARPS_PER_SM, INFO_PAIRS_PER_LAUNCH, INFO_TMEM_COLUMNS, INFO_EDGE_THRESHOLDS = 1, 2, 3, 4
INFO_KERNEL_SHAPE, INFO_ROW_RUNS = 5, 6
# INFO_KERNEL_SHAPE codes (enum sm_shape): bit-sliced = SHAPE_BITSLICE | half | flags, direct = SHAPE_DIRECT
(SHAPE_HALF, SHAPE_TWO_WORDS, SHAPE_SEG8, SHAPE_C2, SHAPE_HP, SHAPE_MULTI, SHAPE_BITSLICE,
 SHAPE_DIRECT) = 0xF, 0x10, 0x20, 0x40, 0x80, 0x100, 0x200, 0x400
(EDGES1, EDGES2, MATCH, SCORE_ALL, SCORE, BEST, WEB, WEB_FILLED, OUTPUT) = range(9)
_PLANE_DTYPE = {EDGES1: np.uint8, EDGES2: np.uint8, MATCH: np.uint8, SCORE_ALL: np.int32,
                SCORE: np.int32, BEST: np.int32, WEB: np.int32, WEB_FILLED: np.int32,
                OUTPUT: np.uint8}
SM_ERR_DEGENERATE = -4

# every symbol include/stereo_b200.h declares (tests/test_abi.py checks the export list)
SYMBOLS = [
    "sm_last_error", "sm_version", "sm_device_count", "sm_host_alloc", "sm_host_free",
    "sm_create", "sm_create_band", "sm_destroy", "sm_set_stream", "sm_set_kernel",
    "sm_synchronize", "sm_upload_f64", "sm_upload_u8", "sm_edges", "sm_set_edges",
    "sm_match_wta", "sm_match_wta_dev", "sm_match_wta_dev_batch", "sm_match_wta_dev_batch16",
    "sm_elapsed_ms", "sm_last_launches",
    "sm_profile_begin", "sm_profile_read", "sm_set_option", "sm_get_info",
    "sm_fill_web_holes", "sm_set_web", "sm_draw_contour_map", "sm_download", "sm_download_web_u8",
    "sm_download_web_u16", "sm_run_batch", "sm_run_batch16", "sm_band_rows",
    "sm_multi_create", "sm_multi_run_batch", "sm_multi_run_batch16", "sm_multi_device_count", "sm_multi_destroy",
    "sm_bands_create", "sm_bands_run", "sm_bands_run16", "sm_bands_destroy",
    "sm_create_range", "sm_create_band_range", "sm_multi_create_range", "sm_bands_create_range",
    "sm_match_wta_dev_batch_ru16", "sm_run_batch_ru16", "sm_multi_run_batch_ru16", "sm_bands_run_ru16",
    "sm_match_wta_dev_batch_sub16", "sm_run_batch_sub16", "sm_multi_run_batch_sub16", "sm_bands_run_sub16",
]


class StereoError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__("libstereo_b200: %s (status %d)" % (msg, code))
        self.code = code


_lib = None


def lib() -> C.CDLL:
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise StereoError(-100, "%s not found: run `make lib` (or __graft_entry__.build())" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        L.sm_last_error.restype = C.c_char_p
        vp, i, d = C.c_void_p, C.c_int, C.c_double
        L.sm_host_alloc.argtypes = [C.POINTER(vp), C.c_size_t]
        L.sm_host_free.argtypes = [vp]
        L.sm_create.argtypes = [C.POINTER(vp), i, i, i, i, i, i]
        L.sm_create_band.argtypes = [C.POINTER(vp), i, i, i, i, i, i, i, i]
        L.sm_create_range.argtypes = [C.POINTER(vp), i, i, i, i, i, i, i]
        L.sm_create_band_range.argtypes = [C.POINTER(vp), i, i, i, i, i, i, i, i, i]
        L.sm_destroy.argtypes = [vp]
        L.sm_set_stream.argtypes = [vp, vp]
        L.sm_set_kernel.argtypes = [vp, i]
        L.sm_set_option.argtypes = [vp, i, i]
        L.sm_get_info.argtypes = [vp, i]
        L.sm_synchronize.argtypes = [vp]
        L.sm_upload_f64.argtypes = [vp, vp, vp]
        L.sm_upload_u8.argtypes = [vp, vp, vp]
        L.sm_edges.argtypes = [vp, d]
        L.sm_set_edges.argtypes = [vp, vp, vp]
        L.sm_match_wta.argtypes = [vp]
        L.sm_match_wta_dev.argtypes = [vp, vp, vp, vp, vp]
        L.sm_match_wta_dev_batch.argtypes = [vp, i, vp, vp, C.c_size_t, vp, vp, C.c_size_t]
        L.sm_match_wta_dev_batch16.argtypes = [vp, i, vp, vp, C.c_size_t, vp, vp, C.c_size_t]
        L.sm_match_wta_dev_batch_ru16.argtypes = [vp, i, vp, vp, C.c_size_t, vp, vp, vp, C.c_size_t]
        L.sm_match_wta_dev_batch_sub16.argtypes = [vp, i, vp, vp, C.c_size_t, vp, vp, vp, C.c_size_t]
        L.sm_elapsed_ms.argtypes = [vp, C.POINTER(C.c_float)]
        L.sm_last_launches.argtypes = [vp]
        L.sm_profile_begin.argtypes = [vp, i]
        L.sm_profile_read.argtypes = [vp, C.POINTER(i), C.POINTER(d), C.POINTER(d)]
        L.sm_fill_web_holes.argtypes = [vp, i]
        L.sm_set_web.argtypes = [vp, vp]
        L.sm_draw_contour_map.argtypes = [vp, i, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
        L.sm_download.argtypes = [vp, i, i, vp]
        L.sm_download_web_u8.argtypes = [vp, vp]
        L.sm_download_web_u16.argtypes = [vp, vp]
        L.sm_run_batch.argtypes = [vp, i, vp, vp, d, vp, i, vp]
        L.sm_run_batch16.argtypes = [vp, i, vp, vp, d, vp, vp]
        L.sm_run_batch_ru16.argtypes = [vp, i, vp, vp, d, vp, vp, vp]
        L.sm_run_batch_sub16.argtypes = [vp, i, vp, vp, d, vp, vp, vp]
        L.sm_band_rows.argtypes = [i, i, i, C.POINTER(i), C.POINTER(i)]
        L.sm_multi_create.argtypes = [C.POINTER(vp), C.POINTER(i), i, i, i, i, i, i]
        L.sm_multi_create_range.argtypes = [C.POINTER(vp), C.POINTER(i), i, i, i, i, i, i, i]
        L.sm_multi_run_batch.argtypes = [vp, i, vp, vp, d, vp, i, vp]
        L.sm_multi_run_batch16.argtypes = [vp, i, vp, vp, d, vp, vp]
        L.sm_multi_run_batch_ru16.argtypes = [vp, i, vp, vp, d, vp, vp, vp]
        L.sm_multi_run_batch_sub16.argtypes = [vp, i, vp, vp, d, vp, vp, vp]
        L.sm_multi_device_count.argtypes = [vp]
        L.sm_multi_destroy.argtypes = [vp]
        L.sm_bands_create.argtypes = [C.POINTER(vp), C.POINTER(i), i, i, i, i, i, i]
        L.sm_bands_create_range.argtypes = [C.POINTER(vp), C.POINTER(i), i, i, i, i, i, i, i]
        L.sm_bands_run.argtypes = [vp, vp, vp, d, vp, vp]
        L.sm_bands_run16.argtypes = [vp, vp, vp, d, vp, vp]
        L.sm_bands_run_ru16.argtypes = [vp, vp, vp, d, vp, vp, vp]
        L.sm_bands_run_sub16.argtypes = [vp, vp, vp, d, vp, vp, vp]
        L.sm_bands_destroy.argtypes = [vp]
        _lib = L
    return _lib


def _check(rc: int) -> int:
    if rc < 0:
        raise StereoError(rc, lib().sm_last_error().decode(errors="replace"))
    return rc


def device_count() -> int:
    return _check(lib().sm_device_count())


def band_rows(height: int, n_bands: int, band: int):
    a, b = C.c_int(), C.c_int()
    _check(lib().sm_band_rows(height, n_bands, band, C.byref(a), C.byref(b)))
    return a.value, b.value


def _ptr(a: np.ndarray) -> C.c_void_p:
    return C.c_void_p(a.ctypes.data)


class PinnedBuffer:
    """Page-locked host memory from sm_host_alloc, viewed as a numpy array."""

    def __init__(self, shape, dtype):
        self.shape, self.dtype = tuple(shape), np.dtype(dtype)
        n = int(np.prod(self.shape)) * self.dtype.itemsize
        p = C.c_void_p()
        _check(lib().sm_host_alloc(C.byref(p), n))
        self._p = p
        buf = (C.c_uint8 * max(n, 1)).from_address(p.value)
        self.array = np.frombuffer(buf, dtype=self.dtype, count=int(np.prod(self.shape))).reshape(self.shape)

    def free(self):
        if self._p is not None:
            self.array = None
            lib().sm_host_free(self._p)
            self._p = None


class StereoContext:
    """One device + stream + frame geometry (an ``sm_ctx``).

    Mirrors the reference's algorithm() (src/stereo.cu:296-347): upload -> edges ->
    match_wta -> fill_web_holes -> draw_contour_map, every stage downloadable.
    ``min_shift``: search the shifts [min_shift, min_shift + num_shifts) (sm_create_band_range); 0 is the
    reference's range.
    """

    def __init__(self, width, height, num_shifts=30, square_width=21, variant=WRAP, device=0,
                 rows=None, kernel=KERNEL_AUTO, min_shift=0):
        self.W, self.H, self.D, self.sw, self.variant = width, height, num_shifts, square_width, variant
        self.min_shift = min_shift
        self.row0, self.row1 = rows if rows is not None else (0, height)
        self._c = C.c_void_p()
        _check(lib().sm_create_band_range(C.byref(self._c), device, width, height, self.row0, self.row1,
                                          min_shift, num_shifts, square_width, variant))
        if kernel != KERNEL_AUTO:
            self.set_kernel(kernel)

    # -- lifetime ------------------------------------------------------------
    def close(self):
        if self._c:
            lib().sm_destroy(self._c)
            self._c = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- configuration -------------------------------------------------------
    def set_kernel(self, kernel):
        _check(lib().sm_set_kernel(self._c, kernel))

    def set_option(self, option, value):
        _check(lib().sm_set_option(self._c, option, int(value)))

    def get_info(self, what):
        return _check(lib().sm_get_info(self._c, what))

    def set_stream(self, cuda_stream: int):
        _check(lib().sm_set_stream(self._c, C.c_void_p(cuda_stream)))

    def synchronize(self):
        _check(lib().sm_synchronize(self._c))

    # -- pipeline ------------------------------------------------------------
    def _frame(self, a, dtype):
        a = np.ascontiguousarray(a, dtype=dtype)
        if a.shape != (self.H, self.W):
            raise ValueError("expected a %dx%d array, got %r" % (self.H, self.W, a.shape))
        return a

    def upload_u8(self, first, second):
        a, b = self._frame(first, np.uint8), self._frame(second, np.uint8)
        _check(lib().sm_upload_u8(self._c, _ptr(a), _ptr(b)))
        self.synchronize()  # numpy temporaries may die after return

    def upload_f64(self, first, second):
        a, b = self._frame(first, np.float64), self._frame(second, np.float64)
        _check(lib().sm_upload_f64(self._c, _ptr(a), _ptr(b)))
        self.synchronize()

    def edges(self, threshold=0.15):
        _check(lib().sm_edges(self._c, threshold))

    def set_edges(self, first_edges, second_edges):
        a, b = self._frame(first_edges, np.uint8), self._frame(second_edges, np.uint8)
        _check(lib().sm_set_edges(self._c, _ptr(a), _ptr(b)))
        self.synchronize()

    def match_wta(self):
        _check(lib().sm_match_wta(self._c))

    def match_wta_dev(self, d_first_edges: int, d_second_edges: int, d_best: int, d_web: int):
        _check(lib().sm_match_wta_dev(self._c, C.c_void_p(d_first_edges), C.c_void_p(d_second_edges),
                                      C.c_void_p(d_best), C.c_void_p(d_web)))

    def match_wta_dev_batch(self, n_pairs: int, d_first_edges: int, d_second_edges: int, edge_stride: int,
                            d_best: int, d_web: int, out_stride: int):
        """n_pairs resident pairs, strides in elements; pack of pair k+1 overlaps the main kernel of pair k."""
        _check(lib().sm_match_wta_dev_batch(self._c, n_pairs, C.c_void_p(d_first_edges), C.c_void_p(d_second_edges),
                                            edge_stride, C.c_void_p(d_best), C.c_void_p(d_web), out_stride))

    def match_wta_dev_batch16(self, n_pairs: int, d_first_edges: int, d_second_edges: int, edge_stride: int,
                              d_best, d_web: int, out_stride: int):
        """match_wta_dev_batch with uint16 outputs written by the hot kernel; d_best may be None (web only)."""
        _check(lib().sm_match_wta_dev_batch16(self._c, n_pairs, C.c_void_p(d_first_edges), C.c_void_p(d_second_edges),
                                              edge_stride, C.c_void_p(d_best or None), C.c_void_p(d_web), out_stride))

    def match_wta_dev_batch_ru16(self, n_pairs: int, d_first_edges: int, d_second_edges: int, edge_stride: int,
                                 d_best, d_web: int, d_runner_up: int, out_stride: int):
        """match_wta_dev_batch16 that also writes each pixel's runner-up score (the second-largest of its scores over
        the shifts; equal to best where shifts tie) to d_runner_up, uint16 with the web's pair stride."""
        _check(lib().sm_match_wta_dev_batch_ru16(self._c, n_pairs, C.c_void_p(d_first_edges),
                                                 C.c_void_p(d_second_edges), edge_stride, C.c_void_p(d_best or None),
                                                 C.c_void_p(d_web), C.c_void_p(d_runner_up), out_stride))

    def match_wta_dev_batch_sub16(self, n_pairs: int, d_first_edges: int, d_second_edges: int, edge_stride: int,
                                  d_best, d_web: int, d_web_sub: int, out_stride: int):
        """match_wta_dev_batch16 that also writes each pixel's web in sixteenths of a shift (16 * web + frac, frac in
        [-8, 7] from a parabola through the scores next to the winner; see the C header) to d_web_sub, uint16 with the
        web's pair stride.  min_shift + num_shifts <= 4095."""
        _check(lib().sm_match_wta_dev_batch_sub16(self._c, n_pairs, C.c_void_p(d_first_edges),
                                                  C.c_void_p(d_second_edges), edge_stride, C.c_void_p(d_best or None),
                                                  C.c_void_p(d_web), C.c_void_p(d_web_sub), out_stride))

    def elapsed_ms(self) -> float:
        ms = C.c_float()
        _check(lib().sm_elapsed_ms(self._c, C.byref(ms)))
        return ms.value

    def last_launches(self) -> int:
        return _check(lib().sm_last_launches(self._c))

    def profile_begin(self, max_calls: int):
        _check(lib().sm_profile_begin(self._c, max_calls))

    def profile_read(self):
        """(calls recorded, pack kernel ms total, main kernel ms total) since profile_begin."""
        n, p, m = C.c_int(), C.c_double(), C.c_double()
        _check(lib().sm_profile_read(self._c, C.byref(n), C.byref(p), C.byref(m)))
        return n.value, p.value, m.value

    def set_web(self, web):
        a = self._frame(web, np.int32)
        _check(lib().sm_set_web(self._c, _ptr(a)))
        self.synchronize()

    def fill_web_holes(self, times=32):
        _check(lib().sm_fill_web_holes(self._c, times))

    def draw_contour_map(self, lines=10):
        mn, mx = C.c_int32(), C.c_int32()
        _check(lib().sm_draw_contour_map(self._c, lines, C.byref(mn), C.byref(mx)))
        return mn.value, mx.value

    def download(self, which, shift=0, out=None):
        dt = _PLANE_DTYPE[which]
        if out is None:
            out = np.zeros((self.H, self.W), dt)
        assert out.dtype == dt and out.shape == (self.H, self.W) and out.flags.c_contiguous
        _check(lib().sm_download(self._c, which, shift, _ptr(out)))
        return out

    def download_web_u8(self, out=None):
        if out is None:
            out = np.zeros((self.H, self.W), np.uint8)
        _check(lib().sm_download_web_u8(self._c, _ptr(out)))
        return out

    def download_web_u16(self, out=None):
        if out is None:
            out = np.zeros((self.H, self.W), np.uint16)
        assert out.dtype == np.uint16 and out.shape == (self.H, self.W) and out.flags.c_contiguous
        _check(lib().sm_download_web_u16(self._c, _ptr(out)))
        return out

    def run_batch(self, first, second, threshold=0.15, web_u8=False, want_best=False, web_out=None, web16=False,
                  want_runner_up=False, want_subpixel=False):
        """first/second: (n, H, W) u8.  Returns web (n, H, W) [and best]: int32, web as uint8 with web_u8, or (web16)
        both as uint16, written by the hot kernel itself.  want_runner_up (web16 only): also each pixel's runner-up
        score, uint16, last in the result: (web, [best], runner_up).  want_subpixel (web16 only, not with
        want_runner_up): also web_sub, the web in sixteenths of a shift, uint16, last: (web, [best], web_sub)."""
        first = np.ascontiguousarray(first, np.uint8)
        second = np.ascontiguousarray(second, np.uint8)
        n = first.shape[0]
        assert first.shape == second.shape == (n, self.H, self.W)
        return _run_batch(self._c, lib().sm_run_batch, lib().sm_run_batch16, lib().sm_run_batch_ru16, first, second,
                          threshold, web_u8, want_best, web_out, web16, want_runner_up, lib().sm_run_batch_sub16,
                          want_subpixel)

    # -- convenience: the reference's whole step 2 on host edge maps -----------
    def match_wta_host(self, first_edges, second_edges):
        self.set_edges(first_edges, second_edges)
        self.match_wta()
        return self.download(BEST), self.download(WEB)


def _check_extras(web16, want_runner_up, want_subpixel):
    if want_runner_up and not web16:
        raise ValueError("want_runner_up needs web16=True (the runner-up comes with 16-bit results only)")
    if want_subpixel and not web16:
        raise ValueError("want_subpixel needs web16=True (web_sub comes with 16-bit results only)")
    if want_subpixel and want_runner_up:
        raise ValueError("want_subpixel and want_runner_up exclude each other")


def _run_batch(handle, run, run16, run_ru, first, second, threshold, web_u8, want_best, web_out, web16,
               want_runner_up=False, run_sub=None, want_subpixel=False):
    """sm_run_batch / sm_multi_run_batch (run), or with web16 their 16-bit entries (run16), or with want_runner_up
    their runner-up entries (run_ru), or with want_subpixel their sub-pixel entries (run_sub)."""
    if web16 and web_u8:
        raise ValueError("web16 and web_u8 exclude each other")
    _check_extras(web16, want_runner_up, want_subpixel)
    n, H, W = first.shape
    dt = np.uint16 if web16 else (np.uint8 if web_u8 else np.int32)
    if web_out is None:
        web_out = np.zeros((n, H, W), dt)
    assert web_out.dtype == dt and web_out.shape == (n, H, W) and web_out.flags.c_contiguous
    best = np.zeros((n, H, W), np.uint16 if web16 else np.int32) if want_best else None
    if want_runner_up:
        ru = np.zeros((n, H, W), np.uint16)
        _check(run_ru(handle, n, _ptr(first), _ptr(second), threshold, _ptr(web_out), _ptr(best) if want_best else None,
                      _ptr(ru)))
        return (web_out, best, ru) if want_best else (web_out, ru)
    if want_subpixel:
        ws = np.zeros((n, H, W), np.uint16)
        _check(run_sub(handle, n, _ptr(first), _ptr(second), threshold, _ptr(web_out), _ptr(best) if want_best else None,
                       _ptr(ws)))
        return (web_out, best, ws) if want_best else (web_out, ws)
    if web16:
        _check(run16(handle, n, _ptr(first), _ptr(second), threshold, _ptr(web_out), _ptr(best) if want_best else None))
    else:
        _check(run(handle, n, _ptr(first), _ptr(second), threshold, _ptr(web_out), int(web_u8),
                   _ptr(best) if want_best else None))
    return (web_out, best) if want_best else web_out


class MultiGpuBatch:
    """sm_multi_*: whole pairs sharded over several GPUs of one box from ONE process (one context and one host
    thread per entry of `devices`); the C counterpart of launching one rank per GPU.  ``min_shift``: as for
    StereoContext."""

    def __init__(self, devices, width, height, num_shifts, square_width, variant=WRAP, min_shift=0):
        self.W, self.H = width, height
        self._m = C.c_void_p()
        arr = (C.c_int * len(devices))(*devices)
        _check(lib().sm_multi_create_range(C.byref(self._m), arr, len(devices), width, height, min_shift, num_shifts,
                                           square_width, variant))

    def run_batch(self, first, second, threshold=0.15, web_u8=False, want_best=False, web_out=None, web16=False,
                  want_runner_up=False, want_subpixel=False):
        first = np.ascontiguousarray(first, np.uint8)
        second = np.ascontiguousarray(second, np.uint8)
        n = first.shape[0]
        assert first.shape == second.shape == (n, self.H, self.W)
        return _run_batch(self._m, lib().sm_multi_run_batch, lib().sm_multi_run_batch16, lib().sm_multi_run_batch_ru16,
                          first, second, threshold, web_u8, want_best, web_out, web16, want_runner_up,
                          lib().sm_multi_run_batch_sub16, want_subpixel)

    def close(self):
        if self._m:
            lib().sm_multi_destroy(self._m)
            self._m = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


class MultiGpuBands:
    """sm_bands_*: ONE pair split into row bands (with replicated halo rows) over several GPUs from one process.
    ``min_shift``: as for StereoContext."""

    def __init__(self, devices, width, height, num_shifts, square_width, variant=WRAP, min_shift=0):
        self.W, self.H = width, height
        self._b = C.c_void_p()
        arr = (C.c_int * len(devices))(*devices)
        _check(lib().sm_bands_create_range(C.byref(self._b), arr, len(devices), width, height, min_shift, num_shifts,
                                           square_width, variant))

    def run(self, first, second, threshold=0.15, want_best=False, web16=False, want_runner_up=False,
            want_subpixel=False):
        """web [and best] of one pair: int32, or uint16 with web16; want_runner_up (web16 only): also the runner-up
        scores, uint16, last in the result: (web, [best], runner_up); want_subpixel (web16 only, not with
        want_runner_up): web_sub instead, the web in sixteenths of a shift: (web, [best], web_sub)."""
        _check_extras(web16, want_runner_up, want_subpixel)
        first = np.ascontiguousarray(first, np.uint8)
        second = np.ascontiguousarray(second, np.uint8)
        assert first.shape == second.shape == (self.H, self.W)
        dt = np.uint16 if web16 else np.int32
        web = np.zeros((self.H, self.W), dt)
        best = np.zeros((self.H, self.W), dt) if want_best else None
        if want_runner_up:
            ru = np.zeros((self.H, self.W), np.uint16)
            _check(lib().sm_bands_run_ru16(self._b, _ptr(first), _ptr(second), threshold, _ptr(web),
                                           _ptr(best) if want_best else None, _ptr(ru)))
            return (web, best, ru) if want_best else (web, ru)
        if want_subpixel:
            ws = np.zeros((self.H, self.W), np.uint16)
            _check(lib().sm_bands_run_sub16(self._b, _ptr(first), _ptr(second), threshold, _ptr(web),
                                            _ptr(best) if want_best else None, _ptr(ws)))
            return (web, best, ws) if want_best else (web, ws)
        run = lib().sm_bands_run16 if web16 else lib().sm_bands_run
        _check(run(self._b, _ptr(first), _ptr(second), threshold, _ptr(web), _ptr(best) if want_best else None))
        return (web, best) if want_best else web

    def close(self):
        if self._b:
            lib().sm_bands_destroy(self._b)
            self._b = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()
