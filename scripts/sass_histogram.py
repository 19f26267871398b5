#!/usr/bin/env python
"""SASS opcode histogram of the tensor-core kernels of libgfrender.so (CPU only: cuobjdump), the static evidence next to the ncu counters:
   python scripts/sass_histogram.py [libgfrender.so] > profiles/r03_sass_opcodes.txt
Per kernel: instruction count, code bytes, and the opcodes that prove the Blackwell path (UTCHMMA = tcgen05.mma, LDTM/STTM = tcgen05.ld/st,
UBLKCP = cp.async.bulk (TMA), LDGSTS = cp.async, UTCBAR = tcgen05.commit, SYNCS = mbarrier, ELECT = elect.sync, USETMAXREG = setmaxnreg),
and the packed (FFMA2 / FADD2 / FMUL2) next to the scalar fp32 arithmetic."""
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
so = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "geneface_b200", "libgfrender.so")
KEY = ("UTCHMMA", "LDTM", "STTM", "UBLKCP", "LDGSTS", "UTCBAR", "SYNCS", "ELECT", "USETMAXREG", "R2UR", "FFMA2", "FADD2", "FMUL2", "FFMA", "FADD", "FMUL", "HADD2", "F2FP", "LDG", "LDS", "STS", "LD", "ST", "LDC", "ATOMS", "RED", "F2I", "I2FP")
txt = subprocess.run(["cuobjdump", "-sass", so], capture_output=True, text=True, check=True).stdout
cur, hist = None, collections.OrderedDict()
for ln in txt.splitlines():
    m = re.search(r"Function : (\S+)", ln)
    if m:
        cur = subprocess.run(["c++filt", m.group(1)], capture_output=True, text=True).stdout.strip().split("(")[0]
        hist[cur] = collections.Counter()
        continue
    m = re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_]+)", ln)
    if m and cur:
        hist[cur][m.group(1)] += 1
want = re.compile(r"k_tc_(amb|sigcol)<false>|k_dense_tc|k_tl_|k_grid_backward_b200<float, [23], 2>|k_field_fp32|k_march_chunk|k_composite_chunk")
for name, h in hist.items():
    if not want.search(name):
        continue
    n = sum(h.values())
    print("%s: %d instructions (%.1f KB)" % (name, n, n * 16 / 1024))
    print("    " + "  ".join("%s %d" % (k, h[k]) for k in KEY if h.get(k)))
    top = ", ".join("%s %d" % kv for kv in h.most_common(8))
    print("    most frequent: " + top)
