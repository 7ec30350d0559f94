#!/usr/bin/env python3
"""Per-kernel SASS mnemonic histogram of the shipped library (cuobjdump -sass): total instructions and the memory /
warp-level mnemonics the profiles quote.      python tools/sass_histogram.py > profiles/rN_sass_histogram.txt"""
import collections
import os
import re
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PICK = ("LD", "ST", "LDG", "STG", "LDS", "STS", "ATOMS", "ATOMG", "RED", "LDGSTS", "UBLKCP", "UTMALDG", "UTMASTG", "SHFL", "VOTE", "MATCH", "REDUX", "LDL", "STL",
        "BAR", "WARPSYNC", "NANOSLEEP", "MEMBAR")


def main():
    lib = os.path.join(ROOT, "zstandard_b200", "libzstdb200.so")
    out = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    kern, hist = None, collections.OrderedDict()
    for line in out.split("\n"):
        m = re.search(r"Function : (\S+)", line)
        if m:
            name = subprocess.run(["c++filt", m.group(1)], capture_output=True, text=True).stdout.strip().split("(")[0]
            kern = hist.setdefault(name, collections.Counter())
            continue
        m = re.match(r"\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P\d+\s+)?([A-Z][A-Z0-9_.]*)", line)
        if m and kern is not None:
            kern["total"] += 1
            op = m.group(1)
            if op.split(".")[0] in PICK:
                kern[op] += 1
    print("SASS mnemonic histogram of the shipped cubin (cuobjdump -sass zstandard_b200/libzstdb200.so), per kernel: total instructions, then selected "
          "memory / warp-level mnemonics")
    for name in sorted(hist):
        h = hist[name]
        print("%-34s total %6d  %s" % (name, h["total"], "  ".join("%s=%d" % (k, v) for k, v in sorted(h.items()) if k != "total")))


if __name__ == "__main__":
    main()
