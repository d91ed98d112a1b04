#!/usr/bin/env python
"""tools/min_shift_time.py -- what a search range that starts above zero costs, on one GPU.

    python tools/min_shift_time.py --parent DIR [--out profiles/min_shift.json] [--repeats 3]

1. `python bench.py --gpus 1 --steps 10 --warmup 3` in DIR (a built checkout of the parent commit) and in this tree,
   alternating, `repeats` times each: the flagship workload's ms per step must not move.
2. The resident batched hot path at 1920x1080, window 9, 64 pairs per call (sm_match_wta_dev_batch on device edge
   maps, CUDA events of the context: the pack kernels overlap the main kernels on a second stream): (m, D) against
   (0, D) for D in 16, 32, 64, 128 and m in 1, 33, 1000.  The modes of one D alternate within each repeat.
3. The batched edge producer k_edges_planes at the same m values (D = 64): its device time per pair under
   torch.profiler inside sm_run_batch calls of 16 pairs (in a run of its own, after the timings above).
4. `sm_edges` on one 1080p pair (D = 64), host clock around calls that end in a synchronise: m = 0 against m = 33,
   whose call also rebuilds the second image's byte map with the byte-map detector k_edges<uint8_t>.
5. The reason for the feature: a synthetic 1080p pair whose disparities lie in [96, 160), searched as (96, 64)
   against (0, 160) -- resident batched time per pair (as in 2) and end to end from pinned host buffers
   (sm_run_batch16, web only, 32 pairs per call), with the known-answer agreement of both.

The card's name and power limit are read in the same run and stored with the numbers.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import stereomatching_b200 as smb  # noqa: E402
from bench import synth_pair  # noqa: E402

THRESHOLD = 0.15
W, H, SW = 1920, 1080, 9


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
    for f in modes.values():  # warm-up
        for _ in range(2):
            f()
    for _ in range(repeats):
        for m, f in modes.items():
            ts = sorted(f() for _ in range(calls))
            per[m].append(ts[len(ts) // 2])
    return {m: stats(v) for m, v in per.items()}


def bench_steps(parent, repeats):
    out = {"parent": [], "this": []}
    for _ in range(repeats):
        for name, tree in (("parent", parent), ("this", ROOT)):
            r = subprocess.run([sys.executable, "bench.py", "--gpus", "1", "--steps", "10", "--warmup", "3"], cwd=tree,
                               capture_output=True, text=True, check=True)
            line = [x for x in r.stdout.splitlines() if x.startswith("{")][-1]
            out[name].append(json.loads(line)["ms_per_step"])
    return {k: {"runs": v, **stats(v)} for k, v in out.items()}


def banded_pair(seed, m, D):
    """bench.py's synthetic pair with every disparity moved up by m: disparities in [m, m + D)."""
    left, _, disp = synth_pair(seed, W, H, D)
    xs = (np.arange(W)[None, :] - m - disp) % W
    return left, np.ascontiguousarray(np.take_along_axis(left, xs, axis=1)), disp


def device_edges(pairs, n):
    import torch
    e1, e2 = [], []
    with smb.StereoContext(W, H, 16, 3) as c:
        for left, right, _ in pairs:
            c.upload_u8(left, right)
            c.edges(THRESHOLD)
            e1.append(c.download(smb.EDGES1))
            e2.append(c.download(smb.EDGES2))
    k = len(pairs)
    return (torch.from_numpy(np.stack([e1[j % k] for j in range(n)])).cuda(),
            torch.from_numpy(np.stack([e2[j % k] for j in range(n)])).cuda())


def resident(ranges, d1, d2, repeats, calls=10):
    """ranges: name -> (m, D).  ms per sm_match_wta_dev_batch call over all pairs of d1 / d2, alternating."""
    import torch
    n = d1.shape[0]
    npix = W * H
    best = torch.empty((n, npix), dtype=torch.int32, device="cuda")
    web = torch.empty_like(best)
    ctxs = {k: smb.StereoContext(W, H, D, SW, min_shift=m) for k, (m, D) in ranges.items()}
    try:
        def call(c):
            c.match_wta_dev_batch(n, d1.data_ptr(), d2.data_ptr(), npix, best.data_ptr(), web.data_ptr(), npix)
            return c.elapsed_ms()

        return alternate({k: (lambda c=c: call(c)) for k, c in ctxs.items()}, repeats, calls)
    finally:
        for c in ctxs.values():
            c.close()


def edges_planes_per_pair(ms, D=64, n=16):
    import torch
    from torch.profiler import ProfilerActivity, profile
    left, right, _ = synth_pair(1234, W, H, D)
    first = np.ascontiguousarray(np.broadcast_to(left, (n, H, W)))
    second = np.ascontiguousarray(np.broadcast_to(right, (n, H, W)))
    out = {}
    for m in ms:
        with smb.StereoContext(W, H, D, SW, min_shift=m) as c:
            for _ in range(2):
                c.run_batch(first, second, THRESHOLD, web16=True)
            torch.cuda.synchronize()
            calls = 5
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(calls):
                    c.run_batch(first, second, THRESHOLD, web16=True)
                torch.cuda.synchronize()
        us = cnt = 0
        for e in prof.key_averages():
            if "k_edges_planes" in e.key:
                us += getattr(e, "device_time_total", None) or e.cuda_time_total
                cnt += e.count
        out["m=%d" % m] = {"us_per_pair": us / (calls * n), "launches": cnt}
    return out


def sm_edges_per_call(repeats, D=64):
    left, right, _ = synth_pair(1234, W, H, D)
    ctxs = {"m=%d" % m: smb.StereoContext(W, H, D, SW, min_shift=m) for m in (0, 33)}
    try:
        for c in ctxs.values():
            c.upload_u8(left, right)

        def call(c):
            t0 = time.perf_counter()
            c.edges(THRESHOLD)
            c.synchronize()
            return (time.perf_counter() - t0) * 1e3

        return alternate({k: (lambda c=c: call(c)) for k, c in ctxs.items()}, repeats, 50)
    finally:
        for c in ctxs.values():
            c.close()


def known_answer(web, disp, m, D):
    half = SW // 2
    tw, th = max(240, 4 * D), 120
    ys, xs = np.mgrid[0:H, 0:W]
    interior = ((xs % tw >= half) & (xs % tw < tw - m - D - half) & (ys % th >= half + 1) & (ys % th < th - half - 1) &
                (xs >= half) & (xs < W - m - D - half) & (ys >= half + 1) & (ys < H - half - 1))
    return float((web[interior] == m + disp[interior] + 1).mean())


def band_case(repeats, n=32):
    pairs = [banded_pair(1234 + 2 * k, 96, 64) for k in range(4)]
    d1, d2 = device_edges(pairs, n)
    res = {"resident_ms_per_call": resident({"(96, 64)": (96, 64), "(0, 160)": (0, 160)}, d1, d2, repeats),
           "pairs_per_call": n}
    del d1, d2
    f, s = smb.PinnedBuffer((n, H, W), np.uint8), smb.PinnedBuffer((n, H, W), np.uint8)
    for k in range(n):
        f.array[k], s.array[k] = pairs[k % 4][0], pairs[k % 4][1]
    web = smb.PinnedBuffer((n, H, W), np.uint16)
    agree = {}
    ctxs = {"(96, 64)": smb.StereoContext(W, H, 64, SW, min_shift=96), "(0, 160)": smb.StereoContext(W, H, 160, SW)}
    try:
        def call(c):
            t0 = time.perf_counter()
            c.run_batch(f.array, s.array, THRESHOLD, web16=True, web_out=web.array)
            return (time.perf_counter() - t0) * 1e3

        res["end_to_end_ms_per_call"] = alternate({k: (lambda c=c: call(c)) for k, c in ctxs.items()}, repeats, 3)
        for k, c in ctxs.items():
            c.run_batch(f.array, s.array, THRESHOLD, web16=True, web_out=web.array)
            agree[k] = known_answer(web.array[0].astype(np.int32), pairs[0][2], 96, 64)
    finally:
        for c in ctxs.values():
            c.close()
        for b in (f, s, web):
            b.free()
    res["known_answer_agreement"] = agree
    for key in ("resident_ms_per_call", "end_to_end_ms_per_call"):
        r = res[key]
        res[key.replace("ms_per_call", "ratio_96_64_over_0_160")] = r["(96, 64)"]["median"] / r["(0, 160)"]["median"]
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[1])
    ap.add_argument("--parent", required=True, help="a built checkout of the parent commit")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "min_shift.json"))
    ap.add_argument("--repeats", type=int, default=3)
    o = ap.parse_args()
    res = {"card": card(), "repeats": o.repeats,
           "note": "ms per call; median, min and max of the repeats' medians; modes alternate within each repeat"}
    res["bench_ms_per_step"] = bench_steps(os.path.abspath(o.parent), o.repeats)
    n = 64
    d1, d2 = device_edges([synth_pair(1234 + 2 * k, W, H, 64) for k in range(4)], n)
    res["resident_1080p"] = {"pairs_per_call": n, "window": SW, "by_D": {}}
    for D in (16, 32, 64, 128):
        r = resident({"m=%d" % m: (m, D) for m in (0, 1, 33, 1000)}, d1, d2, o.repeats)
        res["resident_1080p"]["by_D"][str(D)] = r
    del d1, d2
    res["sm_edges_1080p_ms_per_call"] = sm_edges_per_call(o.repeats)
    res["band_96_160"] = band_case(o.repeats)
    res["edges_planes_1080p"] = edges_planes_per_pair((0, 1, 33, 1000))
    res["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(o.out)), exist_ok=True)
    with open(o.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
