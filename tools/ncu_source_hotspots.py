#!/usr/bin/env python
"""Source-level hot spots of the hot kernels out of an `ncu --set full --import-source on` capture (library built with
-lineinfo): per kernel the source lines that collect the most warp-stall samples, with the warp instructions they execute and
their dominant stall reasons.  Runs where the report is (no GPU needed):

  python tools/ncu_source_hotspots.py gpurun_out/r02_full.ncu-rep > profiles/r02_source_hotspots.md
"""
import csv
import io
import subprocess
import sys

KERNELS = [("k_onesweep (the first one captured: <8, no gather, one-shot>, a depth-sort pass)", "regex:k_onesweep"),
           ("k_raster (default instantiation)", "regex:k_raster"), ("k_calc_view<Norm6 SH, fused cull>", "regex:k_calc_view"),
           ("k_bin_emit", "regex:k_bin_emit"), ("k_calc_distances", "regex:k_calc_distances")]
TOP = 12


def rows_of(report, kernel):
    out = subprocess.run(["ncu", "-i", report, "--page", "source", "--print-source", "cuda,sass", "--csv", "--kernel-name", kernel, "--launch-count", "1"],
                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True).stdout
    files, cur, header = [], None, None
    for rec in csv.reader(io.StringIO(out)):
        if not rec:
            continue
        if rec[0] == "File Path":
            cur = {"file": rec[1], "lines": []}
            files.append(cur)
        elif rec[0] == "Line No":
            header = rec
        elif cur is not None and header and rec[0].strip().isdigit():
            cur["lines"].append(dict(zip(header[:2] + ["_addr", "_sass"] + header[4:], rec)))
    return files


def num(x):
    try:
        return float(x)
    except ValueError:
        return 0.0


def main():
    report = sys.argv[1]
    print("# source-level hot spots of `%s`\n" % report.split("/")[-1])
    print("`ncu --page source --print-source cuda,sass` of the capture summarised in `r02_ncu_summary.md` (the 33 MB report itself stays in scratch), aggregated per source line (first launch of each kernel;")
    print("stall samples are the sampler's, share = of the kernel's samples; warp-instr = `Instructions Executed`).  Line numbers are")
    print("those of the sources embedded in the capture (`--import-source on`), which later edits may have shifted by a few lines.\n")
    for title, kern in KERNELS:
        files = rows_of(report, kern)
        lines = [(f["file"].split("/")[-1], l) for f in files for l in f["lines"]]
        if not lines:
            continue
        total = sum(num(l["# Samples"]) for _f, l in lines) or 1.0
        instr = sum(num(l["Instructions Executed"]) for _f, l in lines) or 1.0
        stall_cols = [c for c in lines[0][1] if c.startswith("stall_") and "Not Issued" not in c]
        print("## %s\n" % title)
        print("%d stall samples, %.1f M warp instructions over the lines with line info.\n" % (total, instr / 1e6))
        print("| file:line | source | samples | warp-instr | top stalls |")
        print("|---|---|---|---|---|")
        for fname, l in sorted(lines, key=lambda t: -num(t[1]["# Samples"]))[:TOP]:
            st = sorted(((num(l[c]), c[6:]) for c in stall_cols), reverse=True)[:3]
            sts = ", ".join("%s %.0f%%" % (n, 100.0 * v / max(1.0, num(l["# Samples"]))) for v, n in st if v > 0)
            src = l["Source"].strip().replace("|", "\\|")
            if len(src) > 110:
                src = src[:107] + "..."
            print("| %s:%s | `%s` | %.1f%% | %.1f%% | %s |" % (fname, l["Line No"], src, 100.0 * num(l["# Samples"]) / total,
                                                         100.0 * num(l["Instructions Executed"]) / instr, sts))
        print()


if __name__ == "__main__":
    main()
