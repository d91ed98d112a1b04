#!/usr/bin/env python
"""tools/sass_budget.py -- static ALU-pipe budget of the hot kernel's two steady blocks, from the SASS of the built
library (no GPU, no profiler).

    python tools/sass_budget.py [--lib stereomatching_b200/libstereo_b200.so] [--kernel 4,2,16,0,0,0]
                                [--family k_bitslice|k_bitslice16|k_bitslice_ru|k_bitslice_sub|k_bitslice_ru_sub] [--json]

`--kernel` names an instantiation by its template arguments HALF,NW,SEG,MULTI,C2,HP (default: config 2,
window 9, 64 shifts), `--family` the output family (default: k_bitslice, the int32 one).  The SASS (`cuobjdump -sass`) is cut into basic blocks; of those,
  - pass A is the steady walk: among the blocks with the most STS (one per H word and centre word of a walk),
    the one with the fewest ALU-pipe instructions (the VALID_ALL walk, without the validity selects);
  - pass B is the steady block: the largest block that reads tensor memory (LDTM), RB rows x NW words.
Both cover one block of RB rows x (strip columns) pixels per warp, so the ALU-pipe thread instructions per pixel of
the steady state are 32 * (A + B) / (RB * strip columns).  The pipe classes are those of profiles/make_traffic.py.
"""
import argparse
import collections
import json
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "profiles"))
from make_traffic import ALU, FMA, LSU  # noqa: E402

INSTR = re.compile(r"/\*([0-9a-f]{4,})\*/\s+(.*?)\s*;")
BRANCHES = ("BRA", "BRX", "JMP", "JMX", "EXIT", "RET", "CALL")


def bits_for(v):
    b = 0
    while (1 << b) <= v:
        b += 1
    return b


FAMILIES = ("k_bitslice", "k_bitslice16", "k_bitslice_ru", "k_bitslice_sub", "k_bitslice_ru_sub")


def mangled(half, nw, seg, multi, c2, hp, family="k_bitslice"):
    return "%dk_bitslice" % len(family) + family[len("k_bitslice"):] + \
        "ILi%dELi%dELi%dELb%dELb%dELb%dE" % (half, nw, seg, multi, c2, hp)


def opcode(text):
    t = text.split()
    if t[0].startswith("@"):
        t = t[1:]
    return t[0].split(".")[0], t


def function_sass(lib, key):
    out = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    body, on = [], False
    for line in out.splitlines():
        if "Function :" in line:
            on = key in line
            continue
        if on:
            m = INSTR.search(line)
            if m:
                body.append((int(m.group(1), 16), m.group(2)))
    if not body:
        raise SystemExit("no function %s in %s" % (key, lib))
    return body


def basic_blocks(body):
    leaders = {body[0][0]}
    for i, (addr, text) in enumerate(body):
        op, t = opcode(text)
        if op in BRANCHES or op == "BSSY":
            for tok in t[1:]:
                tok = tok.rstrip(",")
                if tok.startswith("0x"):
                    leaders.add(int(tok, 16))
        if op in BRANCHES and i + 1 < len(body):
            leaders.add(body[i + 1][0])
    blocks, cur = [], []
    for addr, text in body:
        if addr in leaders and cur:
            blocks.append(cur)
            cur = []
        cur.append(opcode(text)[0])
    blocks.append(cur)
    return [collections.Counter(b) for b in blocks]


def classes(ops):
    alu = sum(v for k, v in ops.items() if k in ALU)
    fma = sum(v for k, v in ops.items() if k in FMA)
    lsu = sum(v for k, v in ops.items() if k in LSU)
    return {"instructions": sum(ops.values()), "alu": alu, "fma": fma, "lsu": lsu,
            "alu_ops": dict(sorted(((k, v) for k, v in ops.items() if k in ALU), key=lambda kv: -kv[1]))}


def budget(lib, args, family="k_bitslice"):
    half, nw, seg, multi, c2, hp = args
    blocks = basic_blocks(function_sass(lib, mangled(*args, family=family)))
    most_sts = max(b["STS"] for b in blocks)
    alu = lambda b: sum(v for k, v in b.items() if k in ALU)  # noqa: E731
    pass_a = min((b for b in blocks if b["STS"] == most_sts), key=alu)
    pass_b = max((b for b in blocks if b["LDTM"]), key=lambda b: sum(b.values()))
    rb = 32 // (nw * (32 // seg))
    strip_cols = 32 * (2 if hp else 1) * (nw if c2 else 1)
    pixels = rb * strip_cols
    a, b = classes(pass_a), classes(pass_b)
    return {"kernel": "%s<%s>" % (family, ",".join(map(str, args))), "library": lib,
            "planes": {"KH": bits_for(2 * half + 1), "PV": bits_for((2 * half + 1) ** 2)},
            "pixels_per_warp_block": pixels, "pass_a": a, "pass_b": b,
            "alu_per_pixel": {"pass_a": 32.0 * a["alu"] / pixels, "pass_b": 32.0 * b["alu"] / pixels,
                              "steady": 32.0 * (a["alu"] + b["alu"]) / pixels}}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[1])
    ap.add_argument("--lib", default=os.path.join(ROOT, "stereomatching_b200", "libstereo_b200.so"),
                    help="built library or cubin")
    ap.add_argument("--kernel", default="4,2,16,0,0,0", help="HALF,NW,SEG,MULTI,C2,HP")
    ap.add_argument("--family", default="k_bitslice", choices=FAMILIES, help="output family")
    ap.add_argument("--json", action="store_true", help="print the result as JSON")
    o = ap.parse_args()
    r = budget(o.lib, tuple(int(x) for x in o.kernel.split(",")), o.family)
    if o.json:
        json.dump(r, sys.stdout, indent=1)
        print()
        return
    print("%s  (%s)" % (r["kernel"], r["library"]))
    print("| steady block | instrs | ALU pipe | FMA pipe | LSU/TMEM | ALU per pixel | ALU opcodes |")
    print("|---|---|---|---|---|---|---|")
    for name in ("pass_a", "pass_b"):
        c = r[name]
        print("| %s | %d | %d | %d | %d | %.2f | %s |" % (name.replace("_", " "), c["instructions"], c["alu"], c["fma"],
                                                           c["lsu"], r["alu_per_pixel"][name],
                                                           ", ".join("%s %d" % kv for kv in c["alu_ops"].items())))
    print("steady ALU-pipe thread instructions per pixel: %.2f (%d pixels per warp block)"
          % (r["alu_per_pixel"]["steady"], r["pixels_per_warp_block"]))


if __name__ == "__main__":
    main()
