#!/usr/bin/env python
"""tools/runner_up_time.py -- the runner-up entries against the 16-bit ones, on one GPU.

    python tools/runner_up_time.py [--out profiles/runner_up.json] [--repeats 5]

Resident (CUDA events of the context, sm_elapsed_ms): sm_match_wta_dev_batch16 against sm_match_wta_dev_batch_ru16,
both with web + best, per pair of a batch at config 2 (1920x1080, 64 shifts, window 9), config 4 (1280x720, 128
shifts, window 21), the reference's defaults (1920x1080, 30 shifts, window 21), 16 shifts at window 9 (half-word
pairs and column pairs), and four geometries whose runner-up kernels spill more than their 16-bit siblings, 64 pairs
each.  Per repeat each entry runs `calls` timed calls after its warm-up, the two
alternating; the spread is that of the repeats' medians.  best / web of the two entries are checked equal.

End to end from pinned host buffers (host clock around calls that return after their downloads): sm_run_batch16
against sm_run_batch_ru16 at config 2 (64 pairs, web + best).

The card's name and power limit are read in the same run and stored with the numbers.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import stereomatching_b200 as smb  # noqa: E402
from bench import synth_pair  # noqa: E402
from web16_time import THRESHOLD, alternate, card, edge_maps  # noqa: E402


def resident(name, W, H, D, sw, n, repeats):
    import torch
    e1, e2 = edge_maps(W, H, D, n)
    d1, d2 = torch.from_numpy(e1).cuda(), torch.from_numpy(e2).cuda()
    npix = W * H
    b16 = torch.empty((n, npix), dtype=torch.int16, device="cuda")
    w16 = torch.empty_like(b16)
    bru, wru, ru = torch.empty_like(b16), torch.empty_like(b16), torch.empty_like(b16)
    torch.cuda.synchronize()
    with smb.StereoContext(W, H, D, sw) as c:
        def u16():
            c.match_wta_dev_batch16(n, d1.data_ptr(), d2.data_ptr(), npix, b16.data_ptr(), w16.data_ptr(), npix)
            return c.elapsed_ms()

        def ru16():
            c.match_wta_dev_batch_ru16(n, d1.data_ptr(), d2.data_ptr(), npix, bru.data_ptr(), wru.data_ptr(),
                                       ru.data_ptr(), npix)
            return c.elapsed_ms()

        calls = 10
        r = alternate({"u16": u16, "ru16": ru16}, repeats, calls)
        shape = {}
        u16()
        shape["u16"] = c.get_info(smb.INFO_KERNEL_SHAPE)
        ru16()
        shape["ru16"] = c.get_info(smb.INFO_KERNEL_SHAPE)
        pairs_per_launch = c.get_info(smb.INFO_PAIRS_PER_LAUNCH)
        c.synchronize()
        same = bool(torch.equal(w16, wru) and torch.equal(b16, bru))
        ru_le_best = bool(((ru.to(torch.int32) & 0xFFFF) <= (bru.to(torch.int32) & 0xFFFF)).all())
    per_pair = {m: {k: v / n for k, v in s.items()} for m, s in r.items()}
    return {"config": name, "W": W, "H": H, "D": D, "sw": sw, "pairs": n, "calls_per_repeat": calls,
            "ms_per_call": r, "ms_per_pair": per_pair,
            "ratio_ru16_to_u16": r["ru16"]["median"] / r["u16"]["median"],
            "shape": {k: hex(v) for k, v in shape.items()}, "pairs_per_launch_after_ru16": pairs_per_launch,
            "best_web_equal": same, "runner_up_le_best": ru_le_best}


def e2e_config2(repeats, n=64):
    W, H, D, sw = 1920, 1080, 64, 9
    pairs = [synth_pair(1234 + 2 * k, W, H, D) for k in range(4)]
    shape = (n, H, W)
    f, s = smb.PinnedBuffer(shape, np.uint8), smb.PinnedBuffer(shape, np.uint8)
    for k in range(n):
        f.array[k], s.array[k] = pairs[k % 4][0], pairs[k % 4][1]
    web = {k: smb.PinnedBuffer(shape, np.uint16) for k in ("u16", "ru16")}
    best = {k: smb.PinnedBuffer(shape, np.uint16) for k in ("u16", "ru16")}
    ru = smb.PinnedBuffer(shape, np.uint16)
    L = smb.lib()
    with smb.StereoContext(W, H, D, sw) as c:
        def call(kind):
            t0 = time.perf_counter()
            if kind == "u16":
                rc = L.sm_run_batch16(c._c, n, f.array.ctypes.data, s.array.ctypes.data, THRESHOLD,
                                      web[kind].array.ctypes.data, best[kind].array.ctypes.data)
            else:
                rc = L.sm_run_batch_ru16(c._c, n, f.array.ctypes.data, s.array.ctypes.data, THRESHOLD,
                                         web[kind].array.ctypes.data, best[kind].array.ctypes.data, ru.array.ctypes.data)
            t = (time.perf_counter() - t0) * 1e3
            assert rc == 0, L.sm_last_error()
            return t

        r = alternate({k: (lambda k=k: call(k)) for k in ("u16", "ru16")}, repeats, 3)
        same = bool(np.array_equal(web["u16"].array, web["ru16"].array) and
                    np.array_equal(best["u16"].array, best["ru16"].array))
    for b in [f, s, ru] + list(web.values()) + list(best.values()):
        b.free()
    return {"config": "config 2 end to end, web + best", "W": W, "H": H, "D": D, "sw": sw, "pairs": n,
            "ms_per_call": r, "ratio_ru16_to_u16": r["ru16"]["median"] / r["u16"]["median"],
            "best_web_equal": same}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[1])
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "runner_up.json"))
    ap.add_argument("--repeats", type=int, default=5)
    o = ap.parse_args()
    res = {"card": card(), "repeats": o.repeats,
           "note": "ms per call (and per pair); median, min and max of the repeats' medians; entries alternate"}
    res["resident"] = [resident("config 2", 1920, 1080, 64, 9, 64, o.repeats),
                       resident("config 4", 1280, 720, 128, 21, 64, o.repeats),
                       resident("reference defaults", 1920, 1080, 30, 21, 64, o.repeats),
                       resident("16 shifts, window 9", 1920, 1080, 16, 9, 64, o.repeats),
                       # instantiations that spill more than their 16-bit siblings (profiles/runner_up.md)
                       resident("64 shifts, window 7", 1920, 1080, 64, 7, 64, o.repeats),
                       resident("64 shifts, window 13", 1920, 1080, 64, 13, 64, o.repeats),
                       resident("16 shifts, window 11", 1920, 1080, 16, 11, 64, o.repeats),
                       resident("129 shifts, window 13", 1280, 720, 129, 13, 64, o.repeats)]
    res["end_to_end"] = [e2e_config2(o.repeats)]
    res["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(o.out)), exist_ok=True)
    with open(o.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
