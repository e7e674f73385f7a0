#!/usr/bin/env python
"""Per-kernel DRAM traffic and time from an `ncu --set full` report -> the small JSON bench.py reads for
`roofline.traffic` and the `*_dram_gbs_physical` fields (so that those numbers come from a committed capture of the
build being measured, not from literals).

  python tools/ncu_kernels_json.py gpurun_out/prof.ncu-rep "capture description" > profiles/r02_kernels.json
"""
import collections
import csv
import json
import subprocess
import sys

UNIT = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
TIME = {"ns": 1e-3, "us": 1.0, "ms": 1e3, "s": 1e6}


def main():
    rep, note = sys.argv[1], (sys.argv[2] if len(sys.argv) > 2 else "")
    out = subprocess.run(["ncu", "-i", rep, "--page", "raw", "--csv"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True).stdout
    rows = list(csv.reader(out.splitlines()))
    hdr, units, data = rows[0], rows[1], rows[2:]
    col = {h: i for i, h in enumerate(hdr)}
    acc = collections.defaultdict(lambda: {"launches": 0, "dram_read": 0.0, "dram_write": 0.0, "time_us": 0.0, "sm_pct": 0.0, "dram_pct": 0.0,
                                           "warp_instr": 0.0, "regs": 0, "grid": ""})
    for d in data:
        if len(d) != len(hdr):
            continue
        full = d[col["Kernel Name"]].split("(")[0].replace("void ", "").replace("gs::", "")
        name = full.split("<")[0]
        if name == "k_onesweep" and "<" in full:   # <BITS, GATHER, PERSIST>: the persistent variant is the bin sort, not the depth sort
            targs = [a.strip() for a in full[full.index("<") + 1:full.rindex(">")].split(",")]
            if len(targs) >= 3 and targs[2] in ("1", "true", "(bool)1"):
                name = "k_onesweep_binsort"
        a = acc[name]

        def val(m, table):
            try:
                return float(d[col[m]].replace(",", "")) * table.get(units[col[m]], 1.0)
            except (KeyError, ValueError):
                return 0.0
        a["launches"] += 1
        a["dram_read"] += val("dram__bytes_read.sum", UNIT)
        a["dram_write"] += val("dram__bytes_write.sum", UNIT)
        a["time_us"] += val("gpu__time_duration.sum", TIME)
        a["sm_pct"] += val("sm__throughput.avg.pct_of_peak_sustained_elapsed", {})
        a["dram_pct"] += val("gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed", {})
        a["warp_instr"] += val("smsp__inst_executed.sum", {})
        try:
            a["regs"] = int(float(d[col["launch__registers_per_thread"]]))
        except (KeyError, ValueError):
            pass
        a["grid"] = d[col["Grid Size"]].replace(" ", "") if "Grid Size" in col else ""
    res = {}
    for name, a in acc.items():
        n = a["launches"]
        res[name] = {"capture": note, "launches_captured": n, "dram_bytes_per_launch": (a["dram_read"] + a["dram_write"]) / n,
                     "dram_read_bytes_per_launch": a["dram_read"] / n, "dram_write_bytes_per_launch": a["dram_write"] / n,
                     "ncu_time_us_per_launch": a["time_us"] / n, "sm_pct": a["sm_pct"] / n, "dram_pct": a["dram_pct"] / n,
                     "warp_instr_per_launch": a["warp_instr"] / n, "registers": a["regs"], "last_grid": a["grid"]}
    json.dump(res, sys.stdout, indent=1, sort_keys=True)
    print()


if __name__ == "__main__":
    main()
