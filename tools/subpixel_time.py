#!/usr/bin/env python
"""tools/subpixel_time.py -- the sub-pixel entries against the 16-bit ones, on one GPU.

    python tools/subpixel_time.py [--out profiles/subpixel.json] [--repeats 5]

Resident (CUDA events of the context, sm_elapsed_ms): sm_match_wta_dev_batch16 against sm_match_wta_dev_batch_sub16,
both with web + best, per pair of a batch at config 2 (1920x1080, 64 shifts, window 9), config 4 (1280x720, 128
shifts, window 21), the reference's defaults (1920x1080, 30 shifts, window 21), 16 shifts at window 9 (half-word
pairs and column pairs), and the four further geometries of tools/runner_up_time.py, 64 pairs each.  Per repeat
each entry runs `calls` timed calls after its warm-up, the two alternating; the spread is that of the repeats'
medians.  best / web of the two entries are checked equal, and web_sub rounds to web.

End to end from pinned host buffers (host clock around calls that return after their downloads): sm_run_batch16
against sm_run_batch_sub16 at config 2 (64 pairs, web + best).

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
    bsub, wsub, ws = torch.empty_like(b16), torch.empty_like(b16), torch.empty_like(b16)
    torch.cuda.synchronize()
    with smb.StereoContext(W, H, D, sw) as c:
        def u16():
            c.match_wta_dev_batch16(n, d1.data_ptr(), d2.data_ptr(), npix, b16.data_ptr(), w16.data_ptr(), npix)
            return c.elapsed_ms()

        def sub16():
            c.match_wta_dev_batch_sub16(n, d1.data_ptr(), d2.data_ptr(), npix, bsub.data_ptr(), wsub.data_ptr(),
                                        ws.data_ptr(), npix)
            return c.elapsed_ms()

        calls = 10
        r = alternate({"u16": u16, "sub16": sub16}, repeats, calls)
        shape = {}
        u16()
        shape["u16"] = c.get_info(smb.INFO_KERNEL_SHAPE)
        sub16()
        shape["sub16"] = c.get_info(smb.INFO_KERNEL_SHAPE)
        pairs_per_launch = c.get_info(smb.INFO_PAIRS_PER_LAUNCH)
        c.synchronize()
        same = bool(torch.equal(w16, wsub) and torch.equal(b16, bsub))
        rounds = bool(torch.equal(((ws.to(torch.int32) & 0xFFFF) + 8) >> 4, wsub.to(torch.int32) & 0xFFFF))
        frac_nonzero = float(((ws.to(torch.int32) & 15) != 0).float().mean())
    per_pair = {m: {k: v / n for k, v in s.items()} for m, s in r.items()}
    return {"config": name, "W": W, "H": H, "D": D, "sw": sw, "pairs": n, "calls_per_repeat": calls,
            "ms_per_call": r, "ms_per_pair": per_pair,
            "ratio_sub16_to_u16": r["sub16"]["median"] / r["u16"]["median"],
            "shape": {k: hex(v) for k, v in shape.items()}, "pairs_per_launch_after_sub16": pairs_per_launch,
            "best_web_equal": same, "web_sub_rounds_to_web": rounds, "share_frac_nonzero": frac_nonzero}


def e2e_config2(repeats, n=64):
    W, H, D, sw = 1920, 1080, 64, 9
    pairs = [synth_pair(1234 + 2 * k, W, H, D) for k in range(4)]
    shape = (n, H, W)
    f, s = smb.PinnedBuffer(shape, np.uint8), smb.PinnedBuffer(shape, np.uint8)
    for k in range(n):
        f.array[k], s.array[k] = pairs[k % 4][0], pairs[k % 4][1]
    web = {k: smb.PinnedBuffer(shape, np.uint16) for k in ("u16", "sub16")}
    best = {k: smb.PinnedBuffer(shape, np.uint16) for k in ("u16", "sub16")}
    ws = smb.PinnedBuffer(shape, np.uint16)
    L = smb.lib()
    with smb.StereoContext(W, H, D, sw) as c:
        def call(kind):
            t0 = time.perf_counter()
            if kind == "u16":
                rc = L.sm_run_batch16(c._c, n, f.array.ctypes.data, s.array.ctypes.data, THRESHOLD,
                                      web[kind].array.ctypes.data, best[kind].array.ctypes.data)
            else:
                rc = L.sm_run_batch_sub16(c._c, n, f.array.ctypes.data, s.array.ctypes.data, THRESHOLD,
                                          web[kind].array.ctypes.data, best[kind].array.ctypes.data, ws.array.ctypes.data)
            t = (time.perf_counter() - t0) * 1e3
            assert rc == 0, L.sm_last_error()
            return t

        r = alternate({k: (lambda k=k: call(k)) for k in ("u16", "sub16")}, repeats, 3)
        same = bool(np.array_equal(web["u16"].array, web["sub16"].array) and
                    np.array_equal(best["u16"].array, best["sub16"].array))
    for b in [f, s, ws] + list(web.values()) + list(best.values()):
        b.free()
    return {"config": "config 2 end to end, web + best", "W": W, "H": H, "D": D, "sw": sw, "pairs": n,
            "ms_per_call": r, "ratio_sub16_to_u16": r["sub16"]["median"] / r["u16"]["median"],
            "best_web_equal": same}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[1])
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "subpixel.json"))
    ap.add_argument("--repeats", type=int, default=5)
    o = ap.parse_args()
    res = {"card": card(), "repeats": o.repeats,
           "note": "ms per call (and per pair); median, min and max of the repeats' medians; entries alternate"}
    res["resident"] = [resident("config 2", 1920, 1080, 64, 9, 64, o.repeats),
                       resident("config 4", 1280, 720, 128, 21, 64, o.repeats),
                       resident("reference defaults", 1920, 1080, 30, 21, 64, o.repeats),
                       resident("16 shifts, window 9", 1920, 1080, 16, 9, 64, o.repeats),
                       # the runner-up measurement's further geometries (tools/runner_up_time.py)
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
