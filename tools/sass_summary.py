#!/usr/bin/env python
"""SASS evidence for the hot kernels: per kernel the static instruction count, the opcode histogram and the instructions
that answer the usual questions (which copy engine stages the raster's records, are the sort's ballots plain VOTEs, how
many IEEE divisions / square roots does view-calc carry), taken from `cuobjdump -sass` of the built library.

  python tools/sass_summary.py > profiles/r02_sass.md
"""
import collections
import re
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
LIB = ROOT / "unitygaussiansplatting_b200" / "libgsplat_b200.so"
WANT = [("k_onesweep<8, gather, one-shot> (depth sort pass 0)", r"k_onesweepILi8ELb1ELb0E"),
        ("k_onesweep<8, no gather, one-shot> (depth sort passes 1-3, slab sorts)", r"k_onesweepILi8ELb0ELb0E"),
        ("k_onesweep<8, no gather, persistent> (the bin sort)", r"k_onesweepILi8ELb0ELb1E"),
        ("k_raster<fp16 ROP, RGBA16F, no extras> (default)", r"k_rasterILb1ELi0ELb0E"),
        ("k_raster<fp16 ROP, RGBA16F, EXTRAS> (selected splats / scene depth test)", r"k_rasterILb1ELi0ELb1E"),
        ("k_calc_view<3, true, false> (Norm6 SH, fused cull: the Medium frame)", r"k_calc_viewILi3ELb1ELb0E"),
        ("k_calc_distances<0>", r"k_calc_distancesILi0E"), ("k_calc_distances<3> (group of 4: slab table)", r"k_calc_distancesILi3E"),
        ("k_compact_order", r"k_compact_order"), ("k_bin_emit", r"k_bin_emit"), ("k_push_slab (peer stores over NVLink)", r"k_push_slab"),
        ("k_wait_slabs", r"k_wait_slabs")]
NOTABLE = ["LDGSTS", "UBLKCP", "SYNCS", "VOTE", "WARPSYNC", "MATCH", "SHFL", "ATOMS", "ATOMG", "RED", "MUFU.RCP", "MUFU.RSQ", "MUFU.SQRT", "MUFU.EX2",
           "LDG.E.128", "LDG.E.64", "STG.E.128", "STG.E.64", "BAR.SYNC", "CALL", "F2FP", "LDS.128", "LDS.64", "STS.64", "STS.128"]


def main():
    out = subprocess.run(["cuobjdump", "-sass", str(LIB)], stdout=subprocess.PIPE, text=True).stdout
    funcs = {}
    name = None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            name = m.group(1)
            funcs[name] = []
        elif name and re.match(r"\s+/\*[0-9a-f]{4}\*/", line):
            funcs[name].append(line)
    print("# SASS summary of `%s` (sm_100a, `cuobjdump -sass`)\n" % LIB.name)
    for title, pat in WANT:
        hit = [k for k in funcs if re.search(pat, k)]
        if not hit:
            print("## %s\n\nnot found\n" % title)
            continue
        body = funcs[hit[0]]
        ops = collections.Counter()
        for l in body:
            m = re.search(r"\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)", l)
            if m:
                ops[m.group(1)] += 1
        print("## %s\n\n`%s` -- %d static instructions\n" % (title, hit[0][:90], sum(ops.values())))
        print("top opcodes: " + ", ".join("%s %d" % kv for kv in ops.most_common(18)) + "\n")
        notes = []
        for n in NOTABLE:
            c = sum(v for k, v in ops.items() if k.startswith(n))
            if c:
                notes.append("%s %d" % (n, c))
        print("notable: " + ", ".join(notes) + "\n")
        ex = [l.strip() for l in body if re.search(r"LDGSTS|UBLKCP|SYNCS|VOTE|WARPSYNC|MUFU", l)][:12]
        if ex:
            print("```\n" + "\n".join(ex) + "\n```\n")


if __name__ == "__main__":
    main()
