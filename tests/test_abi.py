"""CPU tests of the C-ABI boundary: the library loads, exports exactly what
include/stereo_b200.h declares, and its host-side logic (no GPU needed) is right."""
import ctypes as C
import os
import re
import subprocess

import pytest

import stereomatching_b200 as smb
from util import ROOT


def _header_symbols():
    text = open(os.path.join(ROOT, "include", "stereo_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(sm_[a-z0-9_]+)\s*\(", text)))


def test_library_is_built_in_tree():
    assert os.path.exists(smb.api.LIB_PATH), "run `make lib` / __graft_entry__.build()"
    assert os.path.dirname(smb.api.LIB_PATH).startswith(ROOT)


def test_header_and_binding_list_the_same_symbols():
    assert _header_symbols() == sorted(smb.SYMBOLS)


def test_library_exports_every_declared_symbol():
    L = smb.lib()
    for name in _header_symbols():
        assert hasattr(L, name), name
    out = subprocess.run(["nm", "-D", "--defined-only", smb.api.LIB_PATH], capture_output=True, text=True)
    if out.returncode == 0:
        exported = set(re.findall(r" T (sm_[a-z0-9_]+)", out.stdout))
        assert set(_header_symbols()) <= exported
        # nothing but the C ABI leaks out with C linkage under the sm_ prefix
        assert exported == set(_header_symbols())


def test_signatures_are_plain_c():
    text = open(os.path.join(ROOT, "include", "stereo_b200.h")).read()
    assert 'extern "C"' in text
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)  # comments may mention them
    for bad in ("torch", "at::", "std::", "Tensor", "#include <cuda"):
        assert bad not in text


def test_version_and_error_string():
    L = smb.lib()
    assert L.sm_version() >> 16 == 1
    assert isinstance(L.sm_last_error(), bytes)


def test_info_items_and_shape_codes_match_the_header():
    """ABI 1.3: SM_INFO_KERNEL_SHAPE / SM_INFO_ROW_RUNS and the sm_shape code bits, as the binding spells them."""
    assert smb.lib().sm_version() == (1 << 16) | 3
    text = open(os.path.join(ROOT, "include", "stereo_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    values = {k: int(v, 0) for k, v in re.findall(r"\b(SM_(?:INFO|SHAPE)_[A-Z0-9_]+)\s*=\s*(0x[0-9A-Fa-f]+|\d+)", text)}
    for name, value in values.items():
        assert getattr(smb.api, name[3:]) == value, name
    assert "SM_INFO_KERNEL_SHAPE" in values and "SM_INFO_ROW_RUNS" in values and "SM_SHAPE_DIRECT" in values
    # the flag bits do not overlap each other or the window half
    bits = [v for k, v in values.items() if k.startswith("SM_SHAPE_")]
    assert sum(bits) == 0x7FF and len(bits) == 8


def test_band_rows_partition():
    for h in (1, 7, 135, 1080, 2160):
        for n in (1, 2, 3, 4, 8):
            if n > h:
                continue
            rows = [smb.band_rows(h, n, b) for b in range(n)]
            assert rows[0][0] == 0 and rows[-1][1] == h
            for (a0, a1), (b0, b1) in zip(rows, rows[1:]):
                assert a1 == b0 and a1 > a0
            sizes = [b - a for a, b in rows]
            assert max(sizes) - min(sizes) <= 1
    with pytest.raises(smb.StereoError):
        smb.band_rows(10, 0, 0)
    with pytest.raises(smb.StereoError):
        smb.band_rows(10, 2, 2)


def test_null_context_is_an_error_not_a_crash():
    L = smb.lib()
    assert L.sm_match_wta(None) == -1
    assert b"NULL context" in L.sm_last_error()
    assert L.sm_destroy(None) == 0


def test_create_validates_arguments_before_touching_the_gpu():
    L = smb.lib()
    ctx = C.c_void_p()
    # argument checks come first, so these fail the same way with or without a GPU
    assert L.sm_create(C.byref(ctx), 0, 0, 10, 30, 21, 0) == -1
    assert L.sm_create(C.byref(ctx), 0, 64, 64, 0, 21, 0) == -1
    assert L.sm_create(C.byref(ctx), 0, 64, 64, 513, 21, 0) == -1
    assert L.sm_create(C.byref(ctx), 0, 64, 64, 30, 64, 0) == -1
    assert L.sm_create(C.byref(ctx), 0, 20, 20, 30, 21, 0) == -1  # stereo.cu:395-398
    assert b"square width must not be higher" in L.sm_last_error()
    assert L.sm_create(C.byref(ctx), 0, 64, 64, 30, 21, 2) == -1
    assert L.sm_create_band(C.byref(ctx), 0, 64, 64, 10, 5, 30, 21, 0) == -1
    assert not ctx.value


def test_product_never_imports_the_oracle():
    """The oracle is test infrastructure; the product package and the host drivers must
    not reference it (a product path through the oracle would void every parity claim)."""
    for base in ("stereomatching_b200", "host", "include", "tools"):
        for dirpath, _, files in os.walk(os.path.join(ROOT, base)):
            if "build" in dirpath.split(os.sep):
                continue
            for f in files:
                if f.endswith((".py", ".c", ".h", ".cu", ".cuh")):
                    src = open(os.path.join(dirpath, f), errors="replace").read()
                    assert "import oracle" not in src and "liboracle" not in src and "oracle/" not in src, (
                        os.path.join(dirpath, f))
