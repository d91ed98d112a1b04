#!/usr/bin/env python
"""bench.py -- the hot path's headline measurement (BASELINE.json: MDE/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

Workload (config.workload): BASELINE.json configs[1] -- synthetic textured pairs
1920x1080 with a known disparity field, window 9x9, 64 shifts (SURVEY 8d generator,
seed 1234 + 2k for pair k).  A "step" is one pass of the hot path (bit-plane pack +
match/box/WTA kernel: u8 edge maps resident in HBM -> i32 best + web resident in HBM)
over a batch of `--pairs` stereo pairs, every pair in its own buffers so the step's
working set is far larger than L2.

  value    whole-job MDE/s (pixels x shifts per second), device-timed, inputs resident
  e2e      the same metric through the C ABI with HOST buffers: sm_run_batch
           (H2D u8 images -> edges -> hot path -> D2H i32 web, a three-stage pipeline over groups
           of pairs) per step, wall clock; e2e.link is the measured PCIe ceiling of that call
  roofline the main kernel against the INT32 issue rate measured on this GPU
           (the path is integer-ALU bound, SURVEY 8d; HBM fraction reported alongside)
  cpu_baseline  the reference's own stereo.c hot path (oracle/_ref) on one host core

--impl reference times the UNMODIFIED reference CPU code (oracle/_ref; one process per
host core, each on its own slab of the same workload).
Multi-GPU (torchrun): whole pairs are sharded over ranks, no collective on the data
path (weak scaling: every rank runs `--pairs` pairs per step).

--dump-outputs DIR writes rank 0's `best` and `web` of the last timed step as DIR/best.npy and
DIR/web.npy (float32), so that two builds can be compared output for output on the same inputs.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

W, H, D, SW = 1920, 1080, 64, 9
THRESHOLD = 0.15
OPS_PER_MDE = 8          # SURVEY 8d: algorithmic integer ops per pixel x shift
BYTES_PER_PIXEL = 10     # 2 u8 edge maps in + i32 web + i32 best out
METRIC = "hot-path throughput (pixels x shifts per second)"


# ------------------------------------------------------------------------------------
# synthetic pairs (SURVEY 8d), vectorised numpy; independent of oracle/
# ------------------------------------------------------------------------------------
def _splitmix64(z):
    z = z + np.uint64(0x9E3779B97F4A7C15)
    z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def synth_pair(seed, w, h, d):
    K = np.uint64(0xD6E8FEB86659FD93)
    with np.errstate(over="ignore"):
        ys, xs = np.meshgrid(np.arange(h, dtype=np.uint64), np.arange(w, dtype=np.uint64), indexing="ij")

        def left_at(x):
            hk = _splitmix64(np.uint64(seed) * K + (ys << np.uint64(20)) + x)
            return np.where(((hk >> np.uint64(8)) & np.uint64(7)) == 0, hk & np.uint64(0xFF),
                            np.uint64(128)).astype(np.uint8)

        tw, th = max(240, 4 * d), 120
        hd = _splitmix64(np.uint64(seed + 1) * K + (ys // np.uint64(th)) * np.uint64(4096) + xs // np.uint64(tw))
        disp = (hd % np.uint64(d)).astype(np.int64)
        xsrc = ((xs.astype(np.int64) - disp) % w).astype(np.uint64)
        return left_at(xs), left_at(xsrc), disp.astype(np.int32)


# ------------------------------------------------------------------------------------
# clocks sampling (B200_PROFILING.md recipe)
# ------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(device), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        rows = [r for (t, r) in self.rows if t0 <= t <= t1 and len(r) >= 8] or \
               [r for (t, r) in self.rows if len(r) >= 8][-3:]
        sm = sorted(float(r[0]) for r in rows if r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in rows if r[1].replace(".", "").isdigit()]
        pw = [float(r[2]) for r in rows if r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in rows for n, v in zip(names, r[4:8]) if v.lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(rows), "reasons": reasons}


# ------------------------------------------------------------------------------------
# CPU legs: the reference (oracle/_ref) or, if that is absent, the oracle port
# ------------------------------------------------------------------------------------
def _cpu_slab(args):
    """One worker: hot path of the reference on a slab of `rows` output rows (+ halo)."""
    seed, rows, variant = args
    import oracle
    half = SW // 2
    left, right, _ = synth_pair(seed, W, rows + 2 * half, D)
    if oracle.ref_available(variant, D):
        ref = oracle.RefLib(variant, D)
        e1, e2 = ref.edges(left, THRESHOLD), ref.edges(right, THRESHOLD)
        t0 = time.perf_counter()
        ref.match_wta(e1, e2, SW)
        return time.perf_counter() - t0, "reference"
    orc = oracle.Oracle()
    e1, e2 = orc.edges(left, THRESHOLD, variant), orc.edges(right, THRESHOLD, variant)
    t0 = time.perf_counter()
    orc.match_wta(e1, e2, D, SW, variant, direct=True)
    return time.perf_counter() - t0, "port"


def cpu_baseline_single_core():
    """stereo.c's hot path (fillup_matches + fillup_scores + find_highest_scoring_shifts)
    on ONE core (the reference is single-threaded), bounded sample."""
    rows = 256
    half = SW // 2
    t, kind = _cpu_slab((1234, rows, 0))
    tg, _ = _cpu_slab((1234, rows, 1))
    mde = W * (rows + 2 * half) * D
    return {"value": mde / t / 1e6, "unit": "MDE/s", "cores": 1, "kind": kind,
            "sample": "one 1920x%d slab of the config-2 pair (D=64, sw=9), wrap variant (stereo.c), %.1f s; "
                      "ghost variant (stereo-ghost.c) on the same slab: %.2f MDE/s" % (rows + 2 * half, t, mde / tg / 1e6),
            "host_cores_total": os.cpu_count()}


def whole_algorithm_baselines(pair, variant):
    """The programs' own `elapsed` line for the whole algorithm() (edges + step 2 + step 3, upload
    excluded) on pair 0 of the workload: the reference's stereo.cu rebuilt for sm_100a
    (oracle/_ref, reported baseline) and this repo's C driver.  Best of 3 runs each."""
    import tempfile

    from PIL import Image
    suffix = "-ghost" if variant == "ghost" else ""
    exes = {"reference_cuda_sm100a": os.path.join(ROOT, "oracle", "_ref", "stereopar%s_D%d" % (suffix, D)),
            "this_repo_driver": os.path.join(ROOT, "timing", "stereopar" + suffix)}
    out = {}
    with tempfile.TemporaryDirectory() as d:
        Image.fromarray(pair[0], "L").save(os.path.join(d, "a.png"))
        Image.fromarray(pair[1], "L").save(os.path.join(d, "b.png"))
        for name, exe in exes.items():
            if not os.path.exists(exe):
                out[name] = None
                continue
            best = None
            for _ in range(3):
                r = subprocess.run([exe, "a.png", "b.png", str(THRESHOLD), str(SW)], cwd=d, capture_output=True,
                                   text=True, env=dict(os.environ, STEREO_NUM_SHIFTS=str(D)))
                f = r.stdout.split()
                if r.returncode == 0 and len(f) >= 15:
                    t = float(f[14])
                    best = t if best is None else min(best, t)
            out[name] = None if best is None else {"elapsed_s": best, "MDE_per_s": W * H * D / best / 1e6}
    out["what"] = ("whole algorithm() on pair 0 (edges + match/WTA + hole filling + contour map), each program's own "
                   "'elapsed' line, best of 3 processes; reference = unmodified stereo%s.cu built by oracle/Makefile "
                   "with -gencode arch=compute_100a,code=sm_100a" % suffix)
    return out


def run_reference_arm(a, rank):
    if rank != 0:
        return
    import multiprocessing as mp
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    rows, half = 24, SW // 2
    ctx = mp.get_context("fork")
    kind = "reference"
    try:  # the library the workers run is loaded here as well, so that the process record shows what ran
        import oracle
        if oracle.ref_available(0, D):
            oracle.RefLib(0, D)
    except OSError:
        pass
    with ctx.Pool(cores) as pool:
        def step(s):
            nonlocal kind
            res = pool.map(_cpu_slab, [(1234 + 2 * (s * cores + k), rows, 0) for k in range(cores)])
            kind = res[0][1]
            return max(r[0] for r in res)  # hot-path time of the slowest worker (inputs prepared untimed)
        for s in range(a.warmup):
            step(s)
        t = sum(step(a.warmup + s) for s in range(a.steps))
    mde_step = cores * W * (rows + 2 * half) * D
    value = mde_step * a.steps / t / 1e6
    sample = ("each step: %d processes (one per host core), each the unmodified stereo.c hot path on its own "
              "1920x%d slab of a config-2 pair (D=64, sw=9, wrap)" % (cores, rows + 2 * half))
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": "MDE/s", "n_gpus": a.gpus,
        "steps": a.steps, "warmup": a.warmup, "ms_per_step": t / a.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": {"workload": "synthetic textured pairs 1920x1080, known disparity, window 9x9, 64 shifts "
                               "(BASELINE configs[1]); CPU sample: " + sample, "variant": "wrap"},
        "cpu_baseline": {"value": value, "unit": "MDE/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "MDE/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }), flush=True)


# ------------------------------------------------------------------------------------
# the B200 arm
# ------------------------------------------------------------------------------------
def bind_rank_to_cpus(local_rank, local_world):
    """Give every rank of the node its own, disjoint slice of the CPUs this job may use, so that eight ranks do not
    all run (and first-touch their pinned staging buffers) on the same cores.  Where NVML knows the CPUs next to the
    GPU the slice is taken from those.  Best effort; returns what was done."""
    try:
        allowed = sorted(os.sched_getaffinity(0))
        near = allowed
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
            words = pynvml.nvmlDeviceGetCpuAffinity(h, (max(allowed) + 64) // 64)
            ideal = [c for c in allowed if (words[c // 64] >> (c % 64)) & 1]
            if len(ideal) >= max(2, len(allowed) // max(local_world, 1)):
                near = ideal
        except Exception:  # noqa: BLE001
            pass
        n = max(1, len(near) // max(local_world, 1))
        mine = near[(local_rank * n) % len(near):][:n] or near
        os.sched_setaffinity(0, mine)
        return "cpus %s (%d of %d allowed)" % (",".join(map(str, mine[:4])) + ("..." if len(mine) > 4 else ""),
                                               len(mine), len(allowed))
    except Exception as e:  # noqa: BLE001
        return "not bound: %s" % type(e).__name__


class Env:
    """Rank bookkeeping: barrier, max over ranks (gloo control plane; the data path has no collective)."""

    def __init__(self, rank, world, local_rank):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.rank, self.world, self.local_rank = rank, world, local_rank
        torch.cuda.set_device(local_rank)
        self.dev = torch.device("cuda", local_rank)
        if world > 1:
            # control plane only (barrier + max of the per-rank time): the data path has no exchange step,
            # so no NCCL communicator is ever needed (SURVEY 8e); gloo keeps stdout to the one JSON line
            dist.init_process_group("gloo")

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def rmax(self, x):
        if self.world > 1:
            t = self.torch.tensor([x], dtype=self.torch.float64)
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
            return float(t.item())
        return x

    def rsum(self, x):
        if self.world > 1:
            t = self.torch.tensor([x], dtype=self.torch.float64)
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
            return float(t.item())
        return x

    def all_true(self, ok):
        return self.rmax(0.0 if ok else 1.0) == 0.0

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def _crc(a):
    import zlib
    return "%08x" % (zlib.crc32(np.ascontiguousarray(a).tobytes()) & 0xFFFFFFFF)


def _golden():
    return json.load(open(os.path.join(ROOT, "tests", "golden", "golden.json")))


DUMP_ELEMENTS = 1 << 22  # per output: 16 MB of float32


def dump_outputs(path, outputs):
    """Write every device tensor of `outputs` as path/<name>.npy in float32 (the values are small integers, exact in
    float32).  An output of more than DUMP_ELEMENTS elements is written as a fixed sample of them: sorted flat
    indices drawn from seed 0, the same in every run with the same arguments."""
    import torch
    os.makedirs(path, exist_ok=True)
    for name, t in outputs.items():
        if t.numel() > DUMP_ELEMENTS:
            idx = np.unique(np.random.default_rng(0).integers(0, t.numel(), DUMP_ELEMENTS))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        np.save(os.path.join(path, name + ".npy"), t.float().cpu().numpy())


def time_batches(env, ctx, stream, run, steps):
    """steps calls of run() on the context's stream, device-timed, max over ranks -> ms per step."""
    torch = env.torch
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    env.barrier()
    ev0.record(stream)
    for _ in range(steps):
        run()
    ev1.record(stream)
    env.barrier()
    return env.rmax(ev0.elapsed_time(ev1)) / steps


def leg_config4_pairs(env, smb, variant_name, npairs=64):
    """BASELINE configs[3]: whole 1280x720 pairs, 128 shifts, window 21 (the reference's default window), sharded
    over the ranks as whole pairs; `npairs` per GPU and step, resident and end to end (u8 web), every distinct
    pair's web checked against the reference's golden CRC."""
    torch = env.torch
    w, h, d, sw = 1280, 720, 128, 21
    g = _golden()
    variant = smb.GHOST if variant_name == "ghost" else smb.WRAP
    keys = ["synth/c4/%d/%s" % (k, variant_name) for k in range(4)]
    pairs = [synth_pair(g[k]["seed"], w, h, d) for k in keys]
    first = np.stack([pairs[k % 4][0] for k in range(npairs)])
    second = np.stack([pairs[k % 4][1] for k in range(npairs)])
    out = {"workload": "%d synthetic 1280x720 pairs per GPU and step, 128 shifts, window 21x21 (BASELINE configs[3]; "
                       "4 distinct pairs, seeds 1234+2k)" % npairs}
    with smb.StereoContext(w, h, d, sw, variant, device=env.local_rank) as c:
        stream = torch.cuda.Stream(device=env.dev)
        c.set_stream(stream.cuda_stream)
        # edge maps resident: detect them once per distinct pair
        e1 = torch.empty((npairs, h, w), dtype=torch.uint8, device=env.dev)
        e2 = torch.empty_like(e1)
        for k in range(4):
            c.upload_u8(pairs[k][0], pairs[k][1])
            c.edges(THRESHOLD)
            e1[k] = torch.from_numpy(c.download(smb.EDGES1)).to(env.dev)
            e2[k] = torch.from_numpy(c.download(smb.EDGES2)).to(env.dev)
        for k in range(4, npairs):
            e1[k], e2[k] = e1[k % 4], e2[k % 4]
        best = torch.empty((npairs, h, w), dtype=torch.int32, device=env.dev)
        web = torch.empty_like(best)
        run = lambda: c.match_wta_dev_batch(npairs, e1.data_ptr(), e2.data_ptr(), h * w, best.data_ptr(),  # noqa: E731
                                            web.data_ptr(), h * w)
        for _ in range(3):
            run()
        ms = time_batches(env, c, stream, run, 5)
        ok = all(_crc(web[k].cpu().numpy()) == g[keys[k % 4]]["web"] and
                 _crc(best[k].cpu().numpy()) == g[keys[k % 4]]["best"] for k in (0, 1, 2, 3, npairs - 1))
        out["resident"] = {"value": env.world * npairs * w * h * d / (ms * 1e-3) / 1e6, "unit": "MDE/s",
                           "us_per_pair": ms * 1e3 / npairs, "pairs_per_s": env.world * npairs / (ms * 1e-3)}
        # end to end: pinned host u8 images -> H2D -> edges -> hot path -> D2H u8 web; four times the pairs per call,
        # so that the fill and drain of the three-stage pipeline weigh as little as in the headline leg
        ne = 4 * npairs
        shape = (ne,) + first.shape[1:]
        hin1, hin2 = smb.PinnedBuffer(shape, np.uint8), smb.PinnedBuffer(shape, np.uint8)
        hweb = smb.PinnedBuffer(shape, np.uint8)
        for k in range(ne):
            hin1.array[k], hin2.array[k] = pairs[k % 4][0], pairs[k % 4][1]
        c.run_batch(hin1.array, hin2.array, THRESHOLD, web_u8=True, web_out=hweb.array)
        env.barrier()
        t0 = time.perf_counter()
        for _ in range(3):
            c.run_batch(hin1.array, hin2.array, THRESHOLD, web_u8=True, web_out=hweb.array)
        env.barrier()
        te = env.rmax(time.perf_counter() - t0) / 3
        ok = ok and all(_crc(hweb.array[k].astype(np.int32)) == g[keys[k % 4]]["web"] for k in range(ne))
        out["e2e"] = {"value": env.world * ne * w * h * d / te / 1e6, "unit": "MDE/s",
                      "pairs_per_s": env.world * ne / te, "pairs_per_step_per_gpu": ne, "api": "sm_run_batch(web_u8=1)",
                      "h2d_bytes_per_step": 2 * ne * w * h, "d2h_bytes_per_step": ne * w * h}
        hin1.free(), hin2.free(), hweb.free()
    out["parity"] = {"equal_reference_golden": env.all_true(ok),
                     "checked": "resident web+best of pairs 0-3 and the last; every e2e web (CRC32 vs tests/golden)"}
    return out


def leg_config3_bands(env, smb, variant_name):
    """BASELINE configs[2]: ONE synthetic 3840x2160 pair, 256 shifts, window 11, as row bands with replicated
    halo rows, one band per rank (strong scaling; the whole frame on one GPU when N = 1).  No exchange step:
    every rank uploads its rows + half+1 halo rows per side and writes only its own rows."""
    torch = env.torch
    w, h, d, sw = 3840, 2160, 256, 11
    g = _golden()["synth/c3/" + variant_name]
    variant = smb.GHOST if variant_name == "ghost" else smb.WRAP
    left, right, _ = synth_pair(g["seed"], w, h, d)
    r0, r1 = smb.band_rows(h, env.world, env.rank)
    pin_l, pin_r = smb.PinnedBuffer((h, w), np.uint8), smb.PinnedBuffer((h, w), np.uint8)
    pin_web = smb.PinnedBuffer((h, w), np.int32)
    pin_l.array[:], pin_r.array[:] = left, right
    out = {"workload": "one synthetic 3840x2160 pair, 256 shifts, window 11x11, %d row band(s) with replicated halo "
                       "rows (BASELINE configs[2])" % env.world, "rows_per_band": r1 - r0}
    with smb.StereoContext(w, h, d, sw, variant, device=env.local_rank, rows=(r0, r1)) as c:
        stream = torch.cuda.Stream(device=env.dev)
        c.set_stream(stream.cuda_stream)
        # resident: whole-frame edge maps on the device (a band context downloads only its own rows, and the
        # band's pack kernel needs the halo rows as well); a step = pack + match/box/WTA of the band
        with smb.StereoContext(w, h, d, sw, variant, device=env.local_rank) as cf:
            cf.upload_u8(pin_l.array, pin_r.array)
            cf.edges(THRESHOLD)
            e1 = torch.from_numpy(cf.download(smb.EDGES1)).to(env.dev)
            e2 = torch.from_numpy(cf.download(smb.EDGES2)).to(env.dev)
        best = torch.empty((h, w), dtype=torch.int32, device=env.dev)
        web = torch.empty_like(best)
        run = lambda: c.match_wta_dev(e1.data_ptr(), e2.data_ptr(), best.data_ptr(), web.data_ptr())  # noqa: E731
        for _ in range(3):
            run()
        ms = time_batches(env, c, stream, run, 10)
        out["resident"] = {"value": w * h * d / (ms * 1e-3) / 1e6, "unit": "MDE/s", "ms_per_frame": ms,
                           "scaling": "strong"}

        def e2e_step():
            c.upload_u8(pin_l.array, pin_r.array), c.edges(THRESHOLD), c.match_wta()
            c.download(smb.WEB, out=pin_web.array)

        e2e_step()
        env.barrier()
        t0 = time.perf_counter()
        for _ in range(5):
            e2e_step()
        env.barrier()
        te = env.rmax(time.perf_counter() - t0) / 5
        out["e2e"] = {"value": w * h * d / te / 1e6, "unit": "MDE/s", "ms_per_frame": te * 1e3,
                      "api": "sm_upload_u8 (band + halo rows) -> sm_edges -> sm_match_wta -> sm_download(SM_WEB) (band rows)"}
        # parity: this rank's rows against the reference's golden CRCs of the 16 row bands of the whole frame
        nb = len(g["web_bands16"])
        mine = [b for b in range(nb) if r0 <= h * b // nb and h * (b + 1) // nb <= r1]
        ok_e2e = len(mine) > 0 and all(_crc(pin_web.array[h * b // nb:h * (b + 1) // nb]) == g["web_bands16"][b] for b in mine)
        ok_res = len(mine) > 0 and all(_crc(web[h * b // nb:h * (b + 1) // nb].cpu().numpy()) == g["web_bands16"][b] for b in mine)
        ok = ok_e2e and ok_res
    out["parity"] = {"bands_equal_reference_golden": env.all_true(ok), "resident": env.all_true(ok_res),
                     "e2e": env.all_true(ok_e2e),
                     "checked": "each rank's rows of web (resident and e2e) vs the per-band CRC32s of the reference's "
                                "whole-frame output (tests/golden synth/c3)"}
    pin_l.free(), pin_r.free(), pin_web.free()
    return out


def run_b200_arm(a, rank, world, local_rank):
    import benchlib
    import stereomatching_b200 as smb

    env = Env(rank, world, local_rank)
    torch = env.torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the hot path has no CPU fallback")
    dev = env.dev
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))
    binding = bind_rank_to_cpus(local_rank, local_world)
    variant = smb.GHOST if a.variant == "ghost" else smb.WRAP
    B, distinct = a.pairs, min(a.pairs, a.distinct)
    gold = _golden()

    # ---- inputs: `distinct` synthetic pairs, edges computed on the device, replicated into B buffers
    seeds = [1234 + 2 * (rank * distinct + k) for k in range(distinct)]
    pairs = [synth_pair(s, W, H, D) for s in seeds]
    ctx = smb.StereoContext(W, H, D, SW, variant, device=local_rank, kernel=a.kernel)
    e1 = torch.empty((B, H, W), dtype=torch.uint8, device=dev)
    e2 = torch.empty((B, H, W), dtype=torch.uint8, device=dev)
    for k in range(distinct):
        ctx.upload_u8(pairs[k][0], pairs[k][1])
        ctx.edges(THRESHOLD)
        e1[k] = torch.from_numpy(ctx.download(smb.EDGES1)).to(dev)
        e2[k] = torch.from_numpy(ctx.download(smb.EDGES2)).to(dev)
    for k in range(distinct, B):
        e1[k] = e1[k % distinct]
        e2[k] = e2[k % distinct]
    best = torch.empty((B, H, W), dtype=torch.int32, device=dev)
    web = torch.empty((B, H, W), dtype=torch.int32, device=dev)
    stream = torch.cuda.Stream(device=dev)  # a created (non-default) stream: the legacy default stream serialises against others
    ctx.set_stream(stream.cuda_stream)
    torch.cuda.synchronize()
    p1, p2, pb, pw = e1.data_ptr(), e2.data_ptr(), best.data_ptr(), web.data_ptr()
    n8, n32 = H * W, H * W * 4

    def step():
        if a.no_overlap:
            for k in range(B):
                ctx.match_wta_dev(p1 + k * n8, p2 + k * n8, pb + k * n32, pw + k * n32)
        else:  # one call per batch: the pack of group k+1 runs beside the main kernel of group k
            ctx.match_wta_dev_batch(B, p1, p2, n8, pb, pw, n8)

    for _ in range(max(a.warmup, 3)):
        step()
    env.barrier()

    # ---- parity on the timed path: EVERY distinct pair of this rank against the reference's golden CRC
    def golden_of(k):
        key = "synth/c2s/%d/wrap" % seeds[k] if a.variant == "wrap" else ("synth/c2/ghost" if seeds[k] == 1234 else None)
        return gold.get(key) if key else None

    def check_webs(get_web, n, what):
        bad, checked = [], 0
        for k in range(n):
            gk = golden_of(k % distinct)
            if gk is None:
                continue
            checked += 1
            if _crc(get_web(k)) != gk["web"]:
                bad.append(k)
        if bad:
            raise SystemExit("bench.py: %s: web of pairs %r differs from the reference's golden CRC" % (what, bad[:8]))
        return checked

    n_checked = check_webs(lambda k: web[k].cpu().numpy(), min(B, 2 * distinct), "resident")
    parity = {"resident_webs_checked": n_checked, "equal_reference_golden": True,
              "golden": "tests/golden/golden.json synth/c2s/<seed>/wrap: CRC32 of web produced by the unmodified stereo.c"}

    # ---- the timed region: K steps, device-timed on the launching stream, max over ranks
    if a.dump_outputs:  # so that what is dumped cannot be left over from the warm-up steps
        best.fill_(-1), web.fill_(-1)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    env.barrier()
    tw0 = time.perf_counter()
    ev0.record(stream)
    for _ in range(a.steps):
        step()
    ev1.record(stream)
    env.barrier()
    tw1 = time.perf_counter()
    ms = env.rmax(ev0.elapsed_time(ev1))
    launches = a.steps * ctx.last_launches()  # per batch call: one pack + one main launch per group of pairs
    clocks = sampler.stop(tw0, tw1) if sampler else None
    if a.dump_outputs and rank == 0:  # before the legs below write the same buffers again
        dump_outputs(a.dump_outputs, {"best": best, "web": web})
    mde_step = B * W * H * D
    value = world * mde_step * a.steps / (ms * 1e-3) / 1e6
    us_pair_tp = ms * 1e3 / a.steps / B

    # ---- sustained: the same step back to back for >= 2 s, its own clocks sample
    sampler2 = ClockSampler(local_rank) if rank == 0 else None
    n_sus = max(1, int(2.2 / max(ms * 1e-3 / a.steps, 1e-4)))
    env.barrier()
    ts0 = time.perf_counter()
    ms_sus = time_batches(env, ctx, stream, step, n_sus)
    ts1 = time.perf_counter()
    clocks_sus = sampler2.stop(ts0, ts1) if sampler2 else None
    sustained = {"value": world * mde_step / (ms_sus * 1e-3) / 1e6, "unit": "MDE/s", "steps": n_sus,
                 "seconds": ms_sus * 1e-3 * n_sus, "us_per_pair": ms_sus * 1e3 / B, "clocks": clocks_sus}

    # the dominant kernel timed ALONE (one pair per call, nothing overlapped)
    niso = min(B, 32)
    ctx.profile_begin(niso)
    for k in range(niso):
        ctx.match_wta_dev(p1 + k * n8, p2 + k * n8, pb + k * n32, pw + k * n32)
    n_iso, pack_ms, main_ms = ctx.profile_read()
    ctx.profile_begin(0)
    # one pair per call as an application with a single stereo pair would run it: pack + dependent main kernel,
    # calls back to back on one stream (no per-kernel events in between), each pair in its own buffers
    nsp = min(B, 64)
    es0, es1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for k in range(4):
        ctx.match_wta_dev(p1 + k * n8, p2 + k * n8, pb + k * n32, pw + k * n32)
    es0.record(stream)
    for k in range(nsp):
        ctx.match_wta_dev(p1 + k * n8, p2 + k * n8, pb + k * n32, pw + k * n32)
    es1.record(stream)
    torch.cuda.synchronize()
    single_us = es0.elapsed_time(es1) * 1e3 / nsp

    # ---- end to end through the C ABI with host buffers -----------------------------------------------------
    # sm_run_batch: pinned host u8 images -> H2D -> edges -> hot path -> D2H web, a three-stage pipeline.  The web
    # comes back in the compact u8 format the ABI offers for num_shifts <= 255 (values 1..64 here); the i32 format
    # (the reference's in-memory type, four times the D2H bytes) is timed alongside.
    Be = min(B, a.e2e_pairs)
    hin1, hin2 = smb.PinnedBuffer((Be, H, W), np.uint8), smb.PinnedBuffer((Be, H, W), np.uint8)
    hweb8 = smb.PinnedBuffer((Be, H, W), np.uint8)
    hweb = smb.PinnedBuffer((Be, H, W), np.int32)
    for k in range(Be):
        hin1.array[k], hin2.array[k] = pairs[k % distinct][0], pairs[k % distinct][1]
    ectx = smb.StereoContext(W, H, D, SW, variant, device=local_rank, kernel=a.kernel)
    e2e_steps = max(3, min(a.steps, 10))

    def time_e2e(u8):
        out = hweb8.array if u8 else hweb.array
        for _ in range(2):
            ectx.run_batch(hin1.array, hin2.array, THRESHOLD, web_u8=u8, web_out=out)
        env.barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            ectx.run_batch(hin1.array, hin2.array, THRESHOLD, web_u8=u8, web_out=out)
        env.barrier()
        te = env.rmax(time.perf_counter() - t0)
        return world * Be * W * H * D * e2e_steps / te / 1e6, ectx.last_launches()

    e2e8_val, e2e_launches = time_e2e(True)
    e2e_val, _ = time_e2e(False)
    parity["e2e_webs_checked"] = check_webs(lambda k: hweb8.array[k].astype(np.int32), Be, "e2e (u8 web)")
    parity["e2e_i32_webs_checked"] = check_webs(lambda k: hweb.array[k], Be, "e2e (i32 web)")
    # the link's own ceiling for those two calls: pinned host<->device copies, both directions at once
    # -- every rank measures its own link while all the others do the same (they share the host's fabric), and the
    # job's ceiling is the sum of the per-rank ceilings
    # under the traffic mix of the call: 2 bytes up per byte down (u8 web), 2 up per 4 down (i32 web)
    h2d_gbs, d2h_gbs, mixes = benchlib.measure_copy_concurrent(local_rank, env.barrier, mixes=((2, 1), (2, 4)))
    (sec8, up8, _), (sec32, up32, _) = mixes
    ceil8 = env.rsum(up8 / (2.0 * W * H) / sec8 * W * H * D / 1e6)      # pairs per round / seconds per round
    ceil32 = env.rsum(up32 / (2.0 * W * H) / sec32 * W * H * D / 1e6)
    h2d_all, d2h_all = env.rsum(h2d_gbs), env.rsum(d2h_gbs)

    # ---- the other sharded configs north_star names, same process, after the headline legs ---------------------
    c4 = leg_config4_pairs(env, smb, a.variant) if not a.no_extra else None
    c3 = leg_config3_bands(env, smb, a.variant) if not a.no_extra else None

    if rank == 0:
        # ---- roofline of the dominant kernel ------------------------------------------------
        main_s = main_ms * 1e-3 / max(n_iso, 1)
        peaks = {m: benchlib.measure_int_peak(local_rank, i) for i, m in
                 enumerate(["iadd3", "lop3", "iadd3+imad", "lop3+imad"])}
        peak = max(peaks.values())  # the dual-pipe issue ceiling: the hardest denominator
        mp_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        hbm_peak, hbm_src = 6650.0, "of fallback (B200_PROFILING.md)"
        if os.path.exists(mp_path):
            hbm_peak, hbm_src = float(json.load(open(mp_path))["hbm_gbs"]), "of measured (MEASURED_PEAKS.json)"
        prof = {}
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp):
            prof = json.load(open(tp))
        traffic = prof.get("main_kernel_dram_bytes_per_pair")
        sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
        n_sms = torch.cuda.get_device_properties(dev).multi_processor_count
        # executed (not algorithmic) work: thread instructions per pair as counted by ncu for the timed region's
        # launch shape (profiles/traffic.json, refreshed per round) / the per-pair time measured live here
        issue = alu_mix = None
        bl = prof.get("batched_launch")
        if bl and "warp_instructions_per_pair" in bl and a.kernel in (0, 2):
            tinstr = bl["warp_instructions_per_pair"] * 32.0
            rate = tinstr / (us_pair_tp * 1e-6) / 1e12
            issue = {"executed_thread_instr_per_pair": tinstr, "achieved": rate, "unit": "T thread-instr/s",
                     "peak": n_sms * 128 * sm_mhz * 1e6 / 1e12, "frac": rate / (n_sms * 128 * sm_mhz * 1e6 / 1e12),
                     "peak_how": "SMs x 4 schedulers x 32 lanes x SM clock under load (one warp instruction per "
                                 "scheduler and cycle)", "source": bl.get("source")}
            alu_rate = bl["alu_pipe_warp_instructions_per_pair"] * 32.0 / (us_pair_tp * 1e-6) / 1e12
            alu_mix = {"achieved": alu_rate, "peak": n_sms * 64 * sm_mhz * 1e6 / 1e12, "unit": "T thread-instr/s",
                       "frac": alu_rate / (n_sms * 64 * sm_mhz * 1e6 / 1e12),
                       "what": "executed ALU-pipe (LOP3/SHF/IADD3/SEL/ISETP...) thread instructions per second / "
                               "(SMs x 64 lanes x SM clock): the pipe that binds this kernel; counts from the ncu "
                               "opcode table of the throughput launch, time from this run's timed region",
                       "alu_pipe_pct_ncu": bl.get("alu_pipe_pct_of_peak_active")}
        ach_iso = OPS_PER_MDE * W * H * D / main_s / 1e12
        ach_tp = OPS_PER_MDE * W * H * D / (us_pair_tp * 1e-6) / 1e12
        roofline = {
            "bound": "int_alu", "kernel": "k_bitslice (bit-sliced match/box/WTA, window ring in tensor memory)",
            "achieved": ach_tp, "peak": peak / 1e3, "unit": "Tiop/s", "frac": ach_tp / (peak / 1e3),
            "frac_throughput": ach_tp / (peak / 1e3), "frac_isolated": ach_iso / (peak / 1e3),
            "durations": {"throughput_us_per_pair": us_pair_tp, "isolated_us_per_launch": main_s * 1e6,
                          "what": "throughput: timed region / pairs (launches of consecutive groups overlap on two "
                                  "streams); isolated: CUDA events around each of %d one-pair launches, nothing overlapped"
                                  % n_iso},
            "traffic": traffic, "issue": issue, "alu_mix": alu_mix,
            "peak_source": "measured live on this GPU (benchlib/peaks.cu), max over instruction mixes %s "
                           "(1e9 thread-instr/s)" % json.dumps({k: round(v) for k, v in peaks.items()}),
            "algorithmic_ops": "%d int ops per pixel x shift (SURVEY 8d) x %d per pair; the kernel is bit-sliced (32 "
                               "shifts per LOP3) and executes about 2.4 thread instructions per pixel x shift, so "
                               "frac > 1 is expected: alu_mix and issue are the utilisation figures" % (OPS_PER_MDE, W * H * D),
            "pack_kernel_us": pack_ms * 1e3 / max(n_iso, 1),
            "hbm": {"achieved": BYTES_PER_PIXEL * W * H / (us_pair_tp * 1e-6) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                    "frac": BYTES_PER_PIXEL * W * H / (us_pair_tp * 1e-6) / 1e9 / hbm_peak, "source": hbm_src,
                    "bytes_per_pair": BYTES_PER_PIXEL * W * H, "duration": "throughput_us_per_pair"},
        }
        cpu = cpu_baseline_single_core() if world == 1 and not a.no_cpu else None
        refcuda = whole_algorithm_baselines(pairs[0], a.variant) if world == 1 and not a.no_cpu else None
        print(json.dumps({
            "metric": METRIC, "value": value, "unit": "MDE/s", "n_gpus": world, "steps": a.steps,
            "warmup": max(a.warmup, 3), "ms_per_step": ms / a.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
            "config": {"workload": "synthetic textured pairs 1920x1080, known disparity, window 9x9, 64 shifts "
                                   "(BASELINE configs[1])", "variant": a.variant, "pairs_per_step_per_gpu": B,
                       "distinct_pairs": distinct, "frames_per_s": value * 1e6 / (W * H * D),
                       "l2": "every pair has its own input and output buffers: %.1f GB per step, far above the "
                             "126 MB L2" % (B * BYTES_PER_PIXEL * W * H / 1e9),
                       "parallelism": "whole pairs per GPU, no collective", "host_binding_rank0": binding,
                       "one_pair_per_call": {"hot_path_us": single_us, "MDE_per_s": W * H * D / single_us,
                                             "what": "sm_match_wta_dev per pair (pack + dependent main kernel), %d calls "
                                                     "back to back on one stream, every pair in its own (cache-cold) buffers, rank 0" % nsp}},
            "clocks": clocks, "gpu_launches": launches, "sustained": sustained,
            "e2e": {"value": e2e8_val, "unit": "MDE/s", "h2d_bytes_per_step": 2 * Be * W * H,
                    "d2h_bytes_per_step": Be * W * H, "pairs_per_step": Be, "steps": e2e_steps,
                    "api": "sm_run_batch(web_u8=1): pinned host u8 images -> H2D -> edges+planes -> hot path -> D2H u8 web "
                           "(values 1..64; the compact result format of the ABI for num_shifts <= 255)",
                    "timer": "host wall clock around synchronised API calls, max over ranks",
                    "frames_per_s": e2e8_val * 1e6 / (W * H * D), "gpu_launches_per_step": e2e_launches,
                    "link": {"h2d_GBps": h2d_gbs, "d2h_GBps": d2h_gbs, "h2d_GBps_all_ranks": h2d_all,
                             "d2h_GBps_all_ranks": d2h_all,
                             "how": "benchlib: pinned copies of up to 256 MB on two free-running streams, mean of 6 "
                                    "rounds, every rank measuring its own link at the same time (after a barrier). "
                                    "h2d_GBps/d2h_GBps: both directions saturated (rank 0's; *_all_ranks: summed). "
                                    "The ceilings time the call's own traffic mix (2 bytes up per byte down for the "
                                    "u8 web, 2 up per 4 down for the i32 web) and sum the per-rank pair rates",
                             "ceiling_MDE_per_s": ceil8, "frac_of_ceiling": e2e8_val / ceil8,
                             "note": "per pair 2 u8 images go up and one u8 web comes down; the slower direction "
                                     "bounds pairs/s, compute overlaps"},
                    "with_i32_web": {"value": e2e_val, "unit": "MDE/s", "d2h_bytes_per_step": 4 * Be * W * H,
                                     "ceiling_MDE_per_s": ceil32, "frac_of_ceiling": e2e_val / ceil32,
                                     "note": "sm_run_batch(web_u8=0): the reference's in-memory type (int *web, "
                                             "stereo.c:196); same values, four bytes per pixel over the link"}},
            "roofline": roofline, "cpu_baseline": cpu, "reference_cuda_baseline": refcuda, "parity": parity,
            "config4_pairs": c4, "config3_bands": c3,
        }), flush=True)
    hin1.free(), hin2.free(), hweb.free(), hweb8.free()
    ctx.close(), ectx.close()
    env.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--pairs", type=int, default=256, help="stereo pairs per step per GPU")
    ap.add_argument("--distinct", type=int, default=16, help="distinct synthetic pairs generated per GPU")
    ap.add_argument("--e2e-pairs", type=int, default=256, help="pairs per end-to-end step per GPU (the resident step's batch)")
    ap.add_argument("--variant", default="wrap", choices=["wrap", "ghost"])
    ap.add_argument("--kernel", type=int, default=0, help="0 auto, 1 direct, 2 bit-sliced")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-overlap", action="store_true", help="one sm_match_wta_dev call per pair (pack not overlapped)")
    ap.add_argument("--no-extra", action="store_true", help="skip the config4_pairs / config3_bands legs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write best.npy and web.npy of the last timed step (float32; above %d elements a fixed "
                         "seeded sample of them) into DIR" % DUMP_ELEMENTS)
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs needs --impl b200 (the reference arm keeps no outputs)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if local_rank == 0:
        import __graft_entry__
        __graft_entry__.ensure_built()  # compile step only; there is no fallback path
    else:  # wait for local rank 0's build on a fresh checkout
        lib = os.path.join(ROOT, "stereomatching_b200", "libstereo_b200.so")
        for _ in range(600):
            if os.path.exists(lib):
                break
            time.sleep(0.5)
    if a.impl == "reference":
        run_reference_arm(a, rank)
    else:
        run_b200_arm(a, rank, world, local_rank)


if __name__ == "__main__":
    main()
