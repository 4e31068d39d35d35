#!/usr/bin/env python
"""SASS opcode histogram of the shipped library: which Blackwell-only instructions it contains (tcgen05.mma -> UTC*MMA,
tcgen05.ld -> LDTM, TMA -> UTMALDG / UTMASTG / UTMAPF, cluster barriers -> UTCBAR, cp.async -> LDGSTS, ...).
usage: python tools/sass_histogram.py [siren_mri_b200/csrc/libsiren_b200.so] > profiles/rNN_sass_opcodes.txt
       python tools/sass_histogram.py --kernel mlp_fused_step [lib]    every opcode of the kernels whose name holds the
                                                                       string (the FP32 pipe mix: FFMA / FFMA2, MOV, ...)"""
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
args = sys.argv[1:]
kernel = None
if args[:1] == ["--kernel"]:
    kernel, args = args[1], args[2:]
lib = args[0] if args else os.path.join(ROOT, "siren_mri_b200", "csrc", "libsiren_b200.so")
sass = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
per_kernel, cur = collections.defaultdict(collections.Counter), None
for ln in sass.splitlines():
    m = re.search(r"Function : (\S+)", ln)
    if m:
        cur = m.group(1)
        continue
    m = re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\d+\s+)?([A-Z][A-Z0-9_]*(?:\.[A-Z0-9_]+)*)", ln)
    if m and cur:
        per_kernel[cur][m.group(1)] += 1
if kernel is not None:
    for k in sorted(per_kernel):
        if kernel in k:
            c = per_kernel[k]
            print("%s  (%d instructions)" % (k[:110], sum(c.values())))
            for op, n in sorted(c.items(), key=lambda t: (-t[1], t[0])):
                print("  %-44s %6d" % (op, n))
    sys.exit(0)
KEYS = ("UTCHMMA", "UTCQMMA", "UTCBAR", "UTCCP", "LDTM", "STTM", "UTMALDG", "UTMASTG", "UTMAPF", "UTMACCTL", "UTMACMDFLUSH",
        "SYNCS", "LDGSTS", "USETMAXREG", "UCGABAR", "MUFU", "RED", "ATOM")
tot = collections.Counter()
for k, c in per_kernel.items():
    for op, n in c.items():
        for key in KEYS:
            if op.startswith(key):
                tot[op] += n
print("library: %s" % os.path.relpath(lib, ROOT))
print("Blackwell / async-proxy opcodes over all kernels (count of SASS instructions):")
for op, n in sorted(tot.items(), key=lambda t: (-t[1], t[0])):
    print("  %-44s %6d" % (op, n))
print()
for k in sorted(per_kernel):
    c = per_kernel[k]
    hits = {op: n for op, n in c.items() if any(op.startswith(key) for key in KEYS[:13])}
    if not hits:
        continue
    print("%s  (%d instructions)" % (k[:110], sum(c.values())))
    print("    " + ", ".join("%s %d" % (op, n) for op, n in sorted(hits.items(), key=lambda t: -t[1])[:14]))
