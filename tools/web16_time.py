#!/usr/bin/env python
"""tools/web16_time.py -- the 16-bit result entries against the int32 (and u8) ones, on one GPU.

    python tools/web16_time.py [--out profiles/web16.json] [--repeats 5]

Resident (CUDA events of the context, sm_elapsed_ms): sm_match_wta_dev_batch (int32 web + best) against
sm_match_wta_dev_batch16 with web + best and with web only, at config 2 (1920x1080, 64 shifts, window 9, 64 pairs),
config 4 (1280x720, 128 shifts, window 21, 64 pairs) and the config 3 frame (3840x2160, 256 shifts, window 11, one
pair).  Per repeat each mode runs `calls` timed calls after its warm-up, the modes alternating; the spread is that of
the repeats' medians.  The 16-bit outputs are checked equal to the int32 ones.

End to end from pinned host buffers (host clock around calls that return after their downloads): sm_run_batch
(int32 web, u8 web) against sm_run_batch16 at config 4 (256 pairs, web only), and sm_bands_run against
sm_bands_run16 on the config 3 frame with one band (web + best).  The webs downloaded end to end (and the bests of
the band runs) are CRC-checked against the reference's (tests/golden/golden.json); the resident outputs are only
compared with the int32 entry's.

The card's name and power limit are read in the same run and stored with the numbers.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import stereomatching_b200 as smb  # noqa: E402
from bench import synth_pair  # noqa: E402

THRESHOLD = 0.15
GOLDEN = json.load(open(os.path.join(ROOT, "tests", "golden", "golden.json")))


def crc(a):
    return "%08x" % (zlib.crc32(np.ascontiguousarray(a).tobytes()) & 0xFFFFFFFF)


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [x.strip() for x in q.stdout.strip().split(",")] if q.returncode == 0 else ("?", "?", "?")
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def stats(xs):
    xs = sorted(xs)
    return {"median": xs[len(xs) // 2], "min": xs[0], "max": xs[-1]}


def alternate(modes, repeats, calls):
    """modes: name -> fn() returning one call's time in ms.  Returns name -> median/min/max of the repeat medians."""
    per = {m: [] for m in modes}
    for m, f in modes.items():  # warm-up
        for _ in range(2):
            f()
    for _ in range(repeats):
        for m, f in modes.items():
            ts = sorted(f() for _ in range(calls))
            per[m].append(ts[len(ts) // 2])
    return {m: stats(v) for m, v in per.items()}


def edge_maps(W, H, D, n, distinct=4):
    """The device edge detector's maps of `distinct` synthetic pairs, repeated to n pairs."""
    e1, e2 = [], []
    with smb.StereoContext(W, H, D, 3) as c:
        for k in range(distinct):
            left, right, _ = synth_pair(1234 + 2 * k, W, H, D)
            c.upload_u8(left, right)
            c.edges(THRESHOLD)
            e1.append(c.download(smb.EDGES1))
            e2.append(c.download(smb.EDGES2))
    return np.stack([e1[k % distinct] for k in range(n)]), np.stack([e2[k % distinct] for k in range(n)])


def resident(name, W, H, D, sw, n, repeats):
    import torch
    e1, e2 = edge_maps(W, H, D, n)
    d1, d2 = torch.from_numpy(e1).cuda(), torch.from_numpy(e2).cuda()
    npix = W * H
    b32 = torch.empty((n, npix), dtype=torch.int32, device="cuda")
    w32 = torch.empty_like(b32)
    b16 = torch.empty((n, npix), dtype=torch.int16, device="cuda")
    w16 = torch.empty_like(b16)
    torch.cuda.synchronize()
    with smb.StereoContext(W, H, D, sw) as c:
        def i32():
            c.match_wta_dev_batch(n, d1.data_ptr(), d2.data_ptr(), npix, b32.data_ptr(), w32.data_ptr(), npix)
            return c.elapsed_ms()

        def u16(best=True):
            c.match_wta_dev_batch16(n, d1.data_ptr(), d2.data_ptr(), npix, b16.data_ptr() if best else None,
                                    w16.data_ptr(), npix)
            return c.elapsed_ms()

        calls = 10
        r = alternate({"i32_web_best": i32, "u16_web_best": u16, "u16_web": lambda: u16(False)}, repeats, calls)
        i32(), u16()
        c.synchronize()
        same = bool(torch.equal(w16.to(torch.int32) & 0xFFFF, w32) and torch.equal(b16.to(torch.int32) & 0xFFFF, b32))
    return {"config": name, "W": W, "H": H, "D": D, "sw": sw, "pairs": n, "calls_per_repeat": calls, "ms_per_call": r,
            "u16_equals_i32": same}


def e2e_config4(repeats, n=256):
    gs = [GOLDEN["synth/c4/%d/wrap" % k] for k in range(4)]
    W, H, D, sw = gs[0]["w"], gs[0]["h"], gs[0]["D"], gs[0]["sw"]
    pairs = [synth_pair(g["seed"], W, H, D) for g in gs]
    shape = (n, H, W)
    f, s = smb.PinnedBuffer(shape, np.uint8), smb.PinnedBuffer(shape, np.uint8)
    for k in range(n):
        f.array[k], s.array[k] = pairs[k % 4][0], pairs[k % 4][1]
    outs = {"i32": smb.PinnedBuffer(shape, np.int32), "u8": smb.PinnedBuffer(shape, np.uint8),
            "u16": smb.PinnedBuffer(shape, np.uint16)}
    with smb.StereoContext(W, H, D, sw) as c:
        def call(kind):
            t0 = time.perf_counter()
            c.run_batch(f.array, s.array, THRESHOLD, web_u8=kind == "u8", web16=kind == "u16", web_out=outs[kind].array)
            return (time.perf_counter() - t0) * 1e3

        r = alternate({k: (lambda k=k: call(k)) for k in outs}, repeats, 3)
        ok = {k: all(crc(o.array[j].astype(np.int32)) == gs[j % 4]["web"] for j in range(n)) for k, o in outs.items()}
    for b in [f, s] + list(outs.values()):
        b.free()
    return {"config": "config 4 end to end", "W": W, "H": H, "D": D, "sw": sw, "pairs": n, "ms_per_call": r,
            "web_equals_reference": ok, "web_bytes_per_pair": {"i32": 4 * W * H, "u8": W * H, "u16": 2 * W * H}}


def e2e_config3_bands(repeats):
    g = GOLDEN["synth/c3/wrap"]
    W, H, D, sw = g["w"], g["h"], g["D"], g["sw"]
    left, right, _ = synth_pair(g["seed"], W, H, D)
    f, s = smb.PinnedBuffer((H, W), np.uint8), smb.PinnedBuffer((H, W), np.uint8)
    f.array[:], s.array[:] = left, right
    outs = {"i32": (smb.PinnedBuffer((H, W), np.int32), smb.PinnedBuffer((H, W), np.int32)),
            "u16": (smb.PinnedBuffer((H, W), np.uint16), smb.PinnedBuffer((H, W), np.uint16))}
    L = smb.lib()
    with smb.MultiGpuBands([0], W, H, D, sw) as b:
        def call(kind):
            web, best = outs[kind]
            run = L.sm_bands_run16 if kind == "u16" else L.sm_bands_run
            t0 = time.perf_counter()
            rc = run(b._b, C.c_void_p(f.array.ctypes.data), C.c_void_p(s.array.ctypes.data), THRESHOLD,
                     C.c_void_p(web.array.ctypes.data), C.c_void_p(best.array.ctypes.data))
            t = (time.perf_counter() - t0) * 1e3
            assert rc == 0, L.sm_last_error()
            return t

        r = alternate({k: (lambda k=k: call(k)) for k in outs}, repeats, 10)
        ok = {k: crc(w.array.astype(np.int32)) == g["web"] and crc(bs.array.astype(np.int32)) == g["best"]
              for k, (w, bs) in outs.items()}
    for buf in [f, s] + [x for pair in outs.values() for x in pair]:
        buf.free()
    return {"config": "config 3 frame, sm_bands_run with one band, web + best", "W": W, "H": H, "D": D, "sw": sw,
            "ms_per_call": r, "equals_reference": ok, "d2h_bytes": {"i32": 8 * W * H, "u16": 4 * W * H}}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[1])
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "web16.json"))
    ap.add_argument("--repeats", type=int, default=5)
    o = ap.parse_args()
    res = {"card": card(), "repeats": o.repeats,
           "note": "ms per call; median, min and max of the repeats' medians; modes alternate within each repeat"}
    res["resident"] = [resident("config 2", 1920, 1080, 64, 9, 64, o.repeats),
                       resident("config 4", 1280, 720, 128, 21, 64, o.repeats),
                       resident("config 3 frame", 3840, 2160, 256, 11, 1, o.repeats)]
    res["end_to_end"] = [e2e_config4(o.repeats), e2e_config3_bands(o.repeats)]
    res["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(o.out)), exist_ok=True)
    with open(o.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
