#!/usr/bin/env python
"""The comparisons with the original project, stored: tests/golden/ref_cases.json.

tests/test_oracle.py compares the oracle array for array with the original's own functions, and
tests/test_gpu_driver.py compares the files of the debug drivers with those of the original's serial
programs.  Both need the original built into oracle/_ref from its sources, which are not part of this
repository.  So every such test first compares with CRC32s stored here (the convention of golden.json),
and makes the live comparison as well whenever oracle/_ref is built.

The stored values are what the oracle computes for those cases, and for the driver files the PPM text the
original's writer makes of those arrays (test_host._ppm_text).  The live comparisons establish that the
oracle equals the original on exactly these cases, and golden.json's CRCs of the original's edges, best
and web pin the overlapping ones (checked below before anything is written).  Regenerate only where the
live comparisons pass:

    python tests/ref_cases.py
"""
import functools
import json
import os
import sys
import zlib

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import oracle  # noqa: E402
from test_host import _ppm_text  # noqa: E402
from util import ROOT, THRESHOLD, load_pair, vname  # noqa: E402

PATH = os.path.join(ROOT, "tests", "golden", "ref_cases.json")
DRIVER_FIXTURES = ["1-240x135", "2-480x270", "3-960x540"]
SHIFT_COUNTS = (16, 64, 128)
WIDE_WINDOWS = [(120, 60, 30, 23), (90, 90, 64, 27), (200, 64, 30, 31), (96, 70, 30, 33), (80, 64, 16, 63),
                (150, 45, 64, 45)]
HOLE_PASSES = (2, 6, 32)
crc = oracle.crc32


@functools.lru_cache(maxsize=1)
def stored():
    with open(PATH) as f:
        return json.load(f)


def build_case(orc, variant):
    """Fixture 1 at 30 shifts: edges, best/web and score/match planes at windows 21 and 6, edges at other thresholds."""
    a, b = load_pair("1-240x135")
    e1, e2 = orc.edges(a, THRESHOLD, variant), orc.edges(b, THRESHOLD, variant)
    out = {"edges1": crc(e1), "edges2": crc(e2)}
    for sw in (21, 6):
        best, web = orc.match_wta(e1, e2, 30, sw, variant)
        out["sw%d/best" % sw], out["sw%d/web" % sw] = crc(best), crc(web)
        for i in (0, 7, 29):
            m, _, s = orc.shift_planes(e1, e2, sw, i, variant)
            out["sw%d/scores%d" % (sw, i)] = crc(s)
            if variant == oracle.WRAP:  # the original's ghost variant keeps no global match planes to compare
                out["sw%d/matches%d" % (sw, i)] = crc(m)
    for thr in (0.0, 0.05, 0.5, 1.0):
        out["edges1/thr%g" % thr] = crc(orc.edges(a, thr, variant))
    return out


def shift_counts_pair(orc, D):
    return orc.synth_pair(5 + D, 200, 64, D)[:2]


def shift_counts_case(orc, variant):
    out = {}
    for D in SHIFT_COUNTS:
        left, right = shift_counts_pair(orc, D)
        e1, e2 = orc.edges(left, THRESHOLD, variant), orc.edges(right, THRESHOLD, variant)
        best, web = orc.match_wta(e1, e2, D, 9, variant)
        out["D%d" % D] = [crc(e1), crc(e2), crc(best), crc(web)]
    return out


def holes_web():
    """A seeded 37x23 web with holes at row ends (see test_fill_web_holes_equals_reference)."""
    rng = np.random.default_rng(5)
    w, h = 37, 23
    web = rng.integers(1, 31, size=(h, w), dtype=np.int32)
    for (y, x) in [(5, w - 1), (7, 0), (9, w - 1), (10, 0), (12, 18), (12, 19), (13, 18)]:
        web[y, x] = 0
    return web


def fill_holes_case(orc):
    web = holes_web()
    return {"times%d" % t: crc(orc.fill_web_holes(web, t)) for t in HOLE_PASSES}


def wide_windows_maps(w, h, sw):
    rng = np.random.default_rng(w + sw)
    le = (rng.random((h, w)) < 0.4).astype(np.uint8)
    re = np.roll(le, 5, axis=1) ^ (rng.random((h, w)) < 0.03).astype(np.uint8)
    return le, re


def wide_windows_case(orc, variant):
    out = {}
    for (w, h, D, sw) in WIDE_WINDOWS:
        best, web = orc.match_wta(*wide_windows_maps(w, h, sw), D, sw, variant)
        out["%dx%d/D%d/sw%d" % (w, h, D, sw)] = [crc(best), crc(web)]
    return out


def driver_ppms(orc, fixture, variant):
    """The 96 PPM files of test/diff.sh for one fixture at the defaults (30 shifts, window 21): name -> text."""
    a, b = load_pair(fixture)
    e1, e2 = orc.edges(a, THRESHOLD, variant), orc.edges(b, THRESHOLD, variant)
    best, web = orc.match_wta(e1, e2, 30, 21, variant)
    out = {"edges-1.ppm": _ppm_text(e1, True), "edges-2.ppm": _ppm_text(e2, True),
           "score_best-0.ppm": _ppm_text(best, False), "web-1.ppm": _ppm_text(web, False),
           "web-2.ppm": _ppm_text(orc.fill_web_holes(web, 32), False)}
    rc, contour = orc.draw_contour_map(web, 10)
    assert rc == 0
    out["output-0.ppm"] = _ppm_text(contour, True)
    for i in range(30):
        m, sa, s = orc.shift_planes(e1, e2, 21, i, variant)
        out["matches-%d.ppm" % i] = _ppm_text(m, True)
        out["score_all-%d.ppm" % i] = _ppm_text(sa, False)
        out["scores-%d.ppm" % i] = _ppm_text(s, False)
    return out


def file_crcs(directory):
    """name -> CRC32 of every file in `directory`."""
    out = {}
    for name in sorted(os.listdir(directory)):
        with open(os.path.join(directory, name), "rb") as f:
            out[name] = "%08x" % (zlib.crc32(f.read()) & 0xFFFFFFFF)
    return out


def main():
    orc = oracle.Oracle()
    with open(os.path.join(ROOT, "tests", "golden", "golden.json")) as f:
        golden = json.load(f)
    out = {}
    for variant in (oracle.WRAP, oracle.GHOST):
        v = vname(variant)
        out["build/" + v] = build_case(orc, variant)
        g = golden["fixture/1-240x135/" + v]
        assert [out["build/" + v][k] for k in ("edges1", "edges2", "sw21/best", "sw21/web")] == \
            [g["edges1"], g["edges2"], g["best"], g["web"]], "the oracle no longer equals the original's CRCs"
        out["shift_counts/" + v] = shift_counts_case(orc, variant)
        out["wide_windows/" + v] = wide_windows_case(orc, variant)
        for fixture in DRIVER_FIXTURES:
            ppms = driver_ppms(orc, fixture, variant)
            out["driver/%s/%s" % (fixture, v)] = {n: "%08x" % (zlib.crc32(t.encode()) & 0xFFFFFFFF)
                                                  for n, t in sorted(ppms.items())}
    out["fill_web_holes"] = fill_holes_case(orc)
    with open(PATH, "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")
    print("wrote %s (%d entries)" % (PATH, len(out)))


if __name__ == "__main__":
    main()
