#!/usr/bin/env python
"""Summarise an `ncu --metrics gpu__time_duration.sum --csv` launch list into per-kernel shares of one step.
A step ends with the SpMV epilogue (k_spmm_fix_to_dense<true>, the one-column instance launched as "spmv_fix_to_dense";
k_spmv_fix_to_dense and k_spmv_to_dense in older captures); the last `--steps` complete steps are averaged.
usage: python profiles/summarize_launches.py gpurun_out/launches.csv [--steps 2] > profiles/launches_rXX.md"""
import collections
import csv
import re
import sys

path = sys.argv[1]
nsteps = int(sys.argv[sys.argv.index("--steps") + 1]) if "--steps" in sys.argv else 2
rows = list(csv.reader(open(path)))
hi = next(i for i, r in enumerate(rows) if r and r[0] == "ID")
hdr = rows[hi]
ki, vi = hdr.index("Kernel Name"), hdr.index("Metric Value")
data = []
for r in rows[hi + 1:]:
    if len(r) > vi:
        name = r[ki].replace("(bool)1", "true").replace("(bool)0", "false")   # template arguments as ncu may print them
        name = re.sub(r"\(.*", "", name).replace("dsa::", "").replace("void ", "")
        data.append((name, float(r[vi].replace(",", "")) / 1e3))
ends = [i for i, (n, _) in enumerate(data) if n.startswith(("k_spmm_fix_to_dense<true>", "k_spmv_fix_to_dense", "k_spmv_to_dense"))]
if len(ends) < nsteps + 1:
    nsteps = max(len(ends) - 1, 1)
lo, hi_ = ends[-nsteps - 1] + 1, ends[-1] + 1
agg = collections.OrderedDict()
for n, us in data[lo:hi_]:
    a = agg.setdefault(n, [0, 0.0])
    a[0] += 1
    a[1] += us
tot = sum(a[1] for a in agg.values())
print(f"# ncu launch list summary: {path}\n")
print(f"{len(data)} launches captured; last {nsteps} steps = launches [{lo}, {hi_}) ; {hi_ - lo} launches, "
      f"{tot / nsteps:.1f} us of kernel time per step (cold-cache, serialised: compare SHARES, not absolutes)\n")
print("| kernel | launches/step | us/step | avg us | share |")
print("|---|---:|---:|---:|---:|")
for n, (c, us) in sorted(agg.items(), key=lambda kv: -kv[1][1]):
    print(f"| {n} | {c / nsteps:.1f} | {us / nsteps:.1f} | {us / c:.1f} | {100 * us / tot:.1f}% |")
