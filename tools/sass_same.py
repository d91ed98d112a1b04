#!/usr/bin/env python
"""tools/sass_same.py -- are the kernels of two built libraries the same instruction for instruction?  No GPU.

    python tools/sass_same.py OTHER.so [stereomatching_b200/libstereo_b200.so] [--pattern REGEX]

Compares the `cuobjdump -sass` instruction text of every function whose name matches --pattern (default: the
int32 and 16-bit bit-sliced families, the direct kernels, k_pack* and k_edges*; not the runner-up family) and
prints how many were compared and which differ.  Exit status 1 if any differs or one is missing.
"""
import argparse
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INSTR = re.compile(r"/\*[0-9a-f]{4,}\*/\s+(.*?)\s*;")
DEFAULT = r"\d+k_bitslice(16)?I|k_direct(16)?E|k_pack|k_edges"


def functions(lib):
    out = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    res, cur = {}, None
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = re.sub(r"_GLOBAL__N__[0-9a-f]+_", "_GLOBAL__N_", m.group(1))  # the anonymous namespace's hash
            res[cur] = []
            continue
        m = INSTR.search(line)
        if cur and m:
            res[cur].append(m.group(1))
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[1])
    ap.add_argument("other")
    ap.add_argument("lib", nargs="?", default=os.path.join(ROOT, "stereomatching_b200", "libstereo_b200.so"))
    ap.add_argument("--pattern", default=DEFAULT)
    o = ap.parse_args()
    a, b = functions(o.other), functions(o.lib)
    names = sorted(n for n in a if re.search(o.pattern, n))
    differ = [n for n in names if a[n] != b.get(n)]
    print("functions compared: %d, differing: %d" % (len(names), len(differ)))
    for n in differ:
        print("  " + n)
    sys.exit(1 if differ or not names else 0)


if __name__ == "__main__":
    main()
