#!/usr/bin/env python
"""Writes profiles/r02_sass_excerpts.txt: per hot kernel of libkbb200.so the SASS mnemonics that evidence the design
(cuobjdump -sass; no GPU needed)."""
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SO = os.path.join(ROOT, "kubebrain_b200", "libkbb200.so")
OUT = os.path.join(ROOT, "profiles", "r02_sass_excerpts.txt")
WANT = ["k_gather", "k_wire_copy", "k_fanout", "k_emitILb0", "k_dir_merge",
        "k_cursor_p2p"]
PATS = ["UBLKCP", "SYNCS", "FENCE", "LDG.E.128", "STG.E.128", "LDS.128", "REDUX", "VOTE", "MATCH", "SHFL", "ATOM", "RED.",
        "NANOSLEEP", "MEMBAR", "CCTL"]

txt = subprocess.run(["cuobjdump", "-sass", SO], capture_output=True, text=True).stdout
funcs = re.split(r"\n\s*Function : ", txt)
with open(OUT, "w") as fo:
    fo.write("SASS excerpts of kubebrain_b200/libkbb200.so (sm_100a), `cuobjdump -sass`, round-2 build (tools/sass_excerpts.py).\n"
             "UBLKCP = cp.async.bulk (TMA 1-D bulk copy; .S.G global->shared, .G.S shared->global), SYNCS = mbarrier operations,\n"
             "FENCE.VIEW.ASYNC = generic->async proxy fence, LDS.128 / LDG.E.128 / STG.E.128 = 16-byte vector accesses,\n"
             "REDUX / VOTE / MATCH / SHFL = warp collectives (segmented latest-revision reduction, group aggregation).\n\n")
    for f in funcs[1:]:
        name = f.split("\n", 1)[0]
        if "k_gather_jobs" in name or not any(w in name for w in WANT):
            continue
        lines = f.split("\n")
        insts = [l for l in lines if re.search(r"/\*[0-9a-f]{4,5}\*/\s+\S", l)]
        counts = {p: sum(p in l for l in insts) for p in PATS}
        fo.write(f"== {name[:150]}\n   instructions: {len(insts)}   " +
                 "  ".join(f"{k}:{v}" for k, v in counts.items() if v) + "\n")
        shown = {}
        for l in insts:
            for p in ("UBLKCP", "SYNCS.ARRIVE", "SYNCS.PHASECHK", "FENCE.VIEW", "REDUX", "MATCH"):
                if p in l and shown.get(p, 0) < 2:
                    shown[p] = shown.get(p, 0) + 1
                    fo.write("     " + re.sub(r"\s+/\* 0x[0-9a-f]+ \*/", "", l.strip())[:120] + "\n")
        fo.write("\n")
    tens = len(re.findall(r"\b(HMMA|UTCMMA|IMMA|QMMA|UTCHMMA|BMMA)\b", txt))
    fo.write(f"tensor-core instructions in the whole library: {tens} (no contraction on this path)\n")
print(open(OUT).read()[:2500])
