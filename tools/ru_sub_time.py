#!/usr/bin/env python
"""tools/ru_sub_time.py -- the entries with both extras (*_ru_sub16) against the runner-up and sub-pixel entries.

    python tools/ru_sub_time.py --static [--parent-lib PARENT/libstereo_b200.so]    (no GPU)
    python tools/ru_sub_time.py [--out profiles/ru_sub.json] [--repeats 5]        (one GPU)

--static compiles the four 16-bit families' translation units with -Xptxas -v (registers and spills of all 94
instantiations of each), counts the pass-B opcodes at config 2 (tools/sass_budget.py) and, with --parent-lib, runs
tools/sass_same.py against a parent build (the default pattern, the runner-up and the sub-pixel functions).  It writes
profiles/ru_sub.json; a GPU run keeps that part and adds its measurements.

The GPU run, resident (CUDA events of the context, sm_elapsed_ms): sm_match_wta_dev_batch16, _ru16, _sub16 and
_ru_sub16, all with web + best, 64 pairs per call, at the workloads of profiles/subpixel.md.  Per repeat each entry
runs `calls` timed calls after its warm-up, the four alternating; the spread is that of the repeats' medians.  The
four outputs of _ru_sub16 are checked equal to those of _ru16 and _sub16.  End to end from pinned host buffers (host
clock around calls that return after their downloads) at config 2: sm_run_batch_ru_sub16 against sm_run_batch_ru16
followed by sm_run_batch_sub16, alternating, outputs checked equal.  The card's name and power limit are read in the
same run.  It writes the JSON to --out and the Markdown beside it.
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
STATIC = os.path.join(ROOT, "profiles", "ru_sub.json")
FAMS = ("k_bitslice16", "k_bitslice_ru", "k_bitslice_sub", "k_bitslice_ru_sub")
WORKLOADS = [("config 2", 1920, 1080, 64, 9), ("config 4", 1280, 720, 128, 21),
             ("reference defaults", 1920, 1080, 30, 21), ("16 shifts, window 9", 1920, 1080, 16, 9),
             ("64 shifts, window 7", 1920, 1080, 64, 7), ("64 shifts, window 13", 1920, 1080, 64, 13),
             ("16 shifts, window 11", 1920, 1080, 16, 11), ("129 shifts, window 13", 1280, 720, 129, 13)]


# ---------------------------------------------------------------------------------
# static: ptxas, SASS opcodes, sass_same
# ---------------------------------------------------------------------------------
def ptxas_table():
    """{family: {"<HALF,NW,SEG,MULTI,C2,HP>": [registers, spill stores, spill loads]}} from nvcc -Xptxas -v."""
    csrc = os.path.join(ROOT, "stereomatching_b200", "csrc")
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        procs = {f: subprocess.Popen(
            ["nvcc", "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC",
             "-I" + os.path.join(ROOT, "include"), "-Xptxas", "-v", "-c", os.path.join(csrc, f + ".cu"),
             "-o", os.path.join(tmp, f + ".o")], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
            for f in FAMS}
        for f, p in procs.items():
            log, _ = p.communicate()
            assert p.returncode == 0, log[-2000:]
            rows, cur = {}, None
            for line in log.splitlines():
                m = re.search(r"Compiling entry function '(\S+)'", line)
                if m:
                    t = re.search(r"\d+%sILi(\d+)ELi(\d+)ELi(\d+)ELb(\d)ELb(\d)ELb(\d)E" % f, m.group(1))
                    cur = "<%s>" % ",".join(t.groups()) if t else None
                    if cur:
                        rows[cur] = [0, 0, 0]
                    continue
                if cur is None:
                    continue
                m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", line)
                if m:
                    rows[cur][1:] = [int(m.group(1)), int(m.group(2))]
                m = re.search(r"Used (\d+) registers", line)
                if m:
                    rows[cur][0] = int(m.group(1))
            out[f] = rows
    return out


def static(parent_lib):
    import sass_budget
    lib = os.path.join(ROOT, "stereomatching_b200", "libstereo_b200.so")
    res = {"ptxas": ptxas_table(), "pass_b_config2": {}, "pass_a_config2": {}}
    for f in FAMS:
        b = sass_budget.budget(lib, (4, 2, 16, 0, 0, 0), f)
        res["pass_b_config2"][f] = {"alu": b["pass_b"]["alu"], "alu_ops": b["pass_b"]["alu_ops"]}
        res["pass_a_config2"][f] = b["pass_a"]["alu"]
    if parent_lib:
        res["sass_same"] = {}
        for pat in (None, "k_bitslice_ru|k_direct16_ruE", "k_bitslice_sub|k_direct16_subE"):
            cmd = [sys.executable, os.path.join(ROOT, "tools", "sass_same.py"), parent_lib] + (["--pattern", pat] if pat else [])
            r = subprocess.run(cmd, capture_output=True, text=True)
            res["sass_same"][pat or "default"] = r.stdout.strip().splitlines()[-1]
    return res


# ---------------------------------------------------------------------------------
# GPU: resident and end to end
# ---------------------------------------------------------------------------------
def resident(name, W, H, D, sw, n, repeats):
    import torch
    import stereomatching_b200 as smb
    from web16_time import alternate, edge_maps
    e1, e2 = edge_maps(W, H, D, n)
    d1, d2 = torch.from_numpy(e1).cuda(), torch.from_numpy(e2).cuda()
    npix = W * H
    buf = lambda: torch.empty((n, npix), dtype=torch.int16, device="cuda")  # noqa: E731
    o = {k: [buf() for _ in range(4)] for k in ("u16", "ru16", "sub16", "ru_sub16")}  # best, web, extra, extra
    torch.cuda.synchronize()
    with smb.StereoContext(W, H, D, sw) as c:
        p = lambda t: t.data_ptr()  # noqa: E731
        a = (n, p(d1), p(d2), npix)
        calls_of = {
            "u16": lambda: c.match_wta_dev_batch16(*a, p(o["u16"][0]), p(o["u16"][1]), npix),
            "ru16": lambda: c.match_wta_dev_batch_ru16(*a, p(o["ru16"][0]), p(o["ru16"][1]), p(o["ru16"][2]), npix),
            "sub16": lambda: c.match_wta_dev_batch_sub16(*a, p(o["sub16"][0]), p(o["sub16"][1]), p(o["sub16"][3]),
                                                         npix),
            "ru_sub16": lambda: c.match_wta_dev_batch_ru_sub16(*a, p(o["ru_sub16"][0]), p(o["ru_sub16"][1]),
                                                               p(o["ru_sub16"][2]), p(o["ru_sub16"][3]), npix)}

        def timed(f):
            return lambda: (f(), c.elapsed_ms())[1]

        calls = 10
        r = alternate({k: timed(f) for k, f in calls_of.items()}, repeats, calls)
        shape, ppl = {}, {}
        for k, f in calls_of.items():
            f()
            shape[k] = hex(c.get_info(smb.INFO_KERNEL_SHAPE))
            ppl[k] = c.get_info(smb.INFO_PAIRS_PER_LAUNCH)
        c.synchronize()
        rs, ru, sub = o["ru_sub16"], o["ru16"], o["sub16"]
        same = bool(all(torch.equal(rs[i], ru[i]) for i in (0, 1, 2)) and
                    all(torch.equal(rs[i], sub[i]) for i in (0, 1, 3)))
    per_pair = {m: {k: v / n for k, v in s.items()} for m, s in r.items()}
    med = {k: v["median"] for k, v in r.items()}
    return {"config": name, "W": W, "H": H, "D": D, "sw": sw, "pairs": n, "calls_per_repeat": calls,
            "ms_per_call": r, "ms_per_pair": per_pair, "shape": shape, "pairs_per_launch": ppl,
            "ratio_ru_sub16_to_u16": med["ru_sub16"] / med["u16"],
            "ratio_ru_sub16_to_ru16_plus_sub16": med["ru_sub16"] / (med["ru16"] + med["sub16"]),
            "outputs_equal_siblings": same}


def e2e_config2(repeats, n=64):
    import stereomatching_b200 as smb
    from bench import synth_pair
    from web16_time import THRESHOLD, alternate
    W, H, D, sw = 1920, 1080, 64, 9
    pairs = [synth_pair(1234 + 2 * k, W, H, D) for k in range(4)]
    shape = (n, H, W)
    f, s = smb.PinnedBuffer(shape, np.uint8), smb.PinnedBuffer(shape, np.uint8)
    for k in range(n):
        f.array[k], s.array[k] = pairs[k % 4][0], pairs[k % 4][1]
    names = ("web", "best", "ru", "sub")
    out = {k: {b: smb.PinnedBuffer(shape, np.uint16) for b in names} for k in ("two", "one")}
    ptr = lambda k, b: out[k][b].array.ctypes.data  # noqa: E731
    L = smb.lib()
    with smb.StereoContext(W, H, D, sw) as c:
        fp, sp = f.array.ctypes.data, s.array.ctypes.data

        def two():
            t0 = time.perf_counter()
            rc = L.sm_run_batch_ru16(c._c, n, fp, sp, THRESHOLD, ptr("two", "web"), ptr("two", "best"),
                                     ptr("two", "ru"))
            rc = rc or L.sm_run_batch_sub16(c._c, n, fp, sp, THRESHOLD, ptr("two", "web"), ptr("two", "best"),
                                            ptr("two", "sub"))
            t = (time.perf_counter() - t0) * 1e3
            assert rc == 0, L.sm_last_error()
            return t

        def one():
            t0 = time.perf_counter()
            rc = L.sm_run_batch_ru_sub16(c._c, n, fp, sp, THRESHOLD, ptr("one", "web"), ptr("one", "best"),
                                         ptr("one", "ru"), ptr("one", "sub"))
            t = (time.perf_counter() - t0) * 1e3
            assert rc == 0, L.sm_last_error()
            return t

        r = alternate({"ru16_then_sub16": two, "ru_sub16": one}, repeats, 3)
        same = bool(all(np.array_equal(out["two"][b].array, out["one"][b].array) for b in names))
    for b in [f, s] + [x for d in out.values() for x in d.values()]:
        b.free()
    return {"config": "config 2 end to end, web + best", "W": W, "H": H, "D": D, "sw": sw, "pairs": n,
            "ms_per_call": r, "ratio": r["ru_sub16"]["median"] / r["ru16_then_sub16"]["median"],
            "outputs_equal_siblings": same}


# ---------------------------------------------------------------------------------
# report
# ---------------------------------------------------------------------------------
def markdown(res):
    L = ["# Runner-up and sub-pixel web from one launch: `k_bitslice_ru_sub`", ""]
    if "resident" in res:
        cd = res["card"]
        L += ["Measured with `tools/ru_sub_time.py` (`profiles/ru_sub.json`) on one **%s** at a **%s** power limit "
              "(max SM clock %s), read in the same run. 64 pairs per call, web + best, %d timed calls per repeat after "
              "warm-up, %d repeats, the entries alternating; median (min–max of the repeats' medians)." % (
                  cd["name"], cd["power_limit"], cd["max_sm_clock"], res["resident"][0]["calls_per_repeat"],
                  res["repeats"]), "",
              "## Resident (CUDA events, µs per pair)", "",
              "| workload | frame | D | window | shape | `*16` | `*_ru16` | `*_sub16` | `*_ru_sub16` | vs ru16 + sub16 "
              "| vs `*16` | outputs equal |", "|---|---|---|---|---|---|---|---|---|---|---|---|"]
        fmt = lambda s: "%.2f (%.2f–%.2f)" % (1e3 * s["median"], 1e3 * s["min"], 1e3 * s["max"])  # noqa: E731
        for w in res["resident"]:
            pp = w["ms_per_pair"]
            L.append("| %s | %dx%d | %d | %d | %s | %s | %s | %s | %s | **%.2f×** | %.2f× | %s |" % (
                w["config"], w["W"], w["H"], w["D"], w["sw"], w["shape"]["ru_sub16"], fmt(pp["u16"]), fmt(pp["ru16"]),
                fmt(pp["sub16"]), fmt(pp["ru_sub16"]), w["ratio_ru_sub16_to_ru16_plus_sub16"],
                w["ratio_ru_sub16_to_u16"], "yes" if w["outputs_equal_siblings"] else "**NO**"))
        e = res["end_to_end"][0]
        L += ["", "End to end at config 2 (64 pairs from pinned host buffers, web + best, host clock around calls that "
              "return after their downloads): `sm_run_batch_ru16` then `sm_run_batch_sub16` %.2f ms, "
              "`sm_run_batch_ru_sub16` %.2f ms per call, **%.2f×**; outputs equal: %s." % (
                  e["ms_per_call"]["ru16_then_sub16"]["median"], e["ms_per_call"]["ru_sub16"]["median"], e["ratio"],
                  "yes" if e["outputs_equal_siblings"] else "**NO**"), ""]
    st = res.get("static")
    if st:
        L += ["## `pass B` ALU-pipe opcodes at config 2 (`<4,2,16,0,0,0>`)", ""]
        for f in FAMS:
            b = st["pass_b_config2"][f]
            ops = ", ".join("%s %d" % kv for kv in sorted(b["alu_ops"].items(), key=lambda kv: -kv[1]))
            L.append("- `%s`: %s = **%d** (pass A %d)" % (f, ops, b["alu"], st["pass_a_config2"][f]))
        L.append("")
        if "sass_same" in st:
            L += ["## Same SASS as the parent", "",
                  "`python tools/sass_same.py PARENT/libstereo_b200.so` (parent built at the parent commit):", ""]
            L += ["- %s: `%s`" % ("default pattern" if k == "default" else "`--pattern '%s'`" % k, v)
                  for k, v in st["sass_same"].items()]
            L.append("")
        L += ["## Registers and spills (`-Xptxas -v`), every instantiation beside its siblings", "",
              "regs / spill stores, loads (bytes).", "",
              "| `<HALF,NW,SEG,MULTI,C2,HP>` | " + " | ".join(FAMS) + " |", "|---" * (len(FAMS) + 1) + "|"]
        key = lambda k: tuple(int(x) for x in k.strip("<>").split(","))  # noqa: E731
        for k in sorted(st["ptxas"]["k_bitslice_ru_sub"], key=key):
            L.append("| %s | " % k + " | ".join("%d / %d, %d" % tuple(st["ptxas"][f].get(k, (0, 0, 0)))
                                                for f in FAMS) + " |")
        L.append("")
    return "\n".join(L)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[1])
    ap.add_argument("--out", default=STATIC)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--static", action="store_true", help="compile-time tables only (no GPU)")
    ap.add_argument("--parent-lib", help="a parent build of libstereo_b200.so for tools/sass_same.py")
    o = ap.parse_args()
    res = {}
    if os.path.exists(STATIC):
        with open(STATIC) as fh:
            res = json.load(fh)
    if o.static:
        res["static"] = static(o.parent_lib)
    else:
        from web16_time import card
        res.update({"card": card(), "repeats": o.repeats,
                    "note": "ms per call (and per pair); median, min and max of the repeats' medians; entries "
                            "alternate"})
        res["resident"] = [resident(*w, 64, o.repeats) for w in WORKLOADS]
        res["end_to_end"] = [e2e_config2(o.repeats)]
        res["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(o.out)), exist_ok=True)
    with open(o.out, "w") as fh:
        json.dump(res, fh, indent=1)
    with open(os.path.splitext(o.out)[0] + ".md", "w") as fh:
        fh.write(markdown(res))
    print(json.dumps({k: v for k, v in res.items() if k != "static"}, indent=1))


if __name__ == "__main__":
    main()
