#!/usr/bin/env python
"""Turn ncu outputs brought back in gpurun_out/ into the small text summaries kept under profiles/.

    python tools/ncu_summary.py launches <launches.csv> <out.txt>      per-kernel launch list (share of step)
    python tools/ncu_summary.py full <prof.ncu-rep> <out.txt> [k3_json] key metrics of each captured launch
"""
import collections
import csv
import json
import subprocess
import sys

KEYS = [
    "gpu__time_duration.sum", "launch__grid_size", "launch__block_size", "launch__registers_per_thread",
    "launch__occupancy_limit_registers", "launch__occupancy_limit_shared_mem", "launch__occupancy_limit_warps",
    "dram__bytes_read.sum", "dram__bytes_write.sum", "gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed",
    "lts__throughput.avg.pct_of_peak_sustained_elapsed", "l1tex__throughput.avg.pct_of_peak_sustained_elapsed",
    "sm__throughput.avg.pct_of_peak_sustained_elapsed", "sm__warps_active.avg.pct_of_peak_sustained_active",
    "smsp__issue_active.avg.pct_of_peak_sustained_active", "smsp__inst_executed.sum",
    "sm__inst_executed_pipe_fma.sum", "sm__inst_executed_pipe_lsu.sum", "sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active",
]


def launches(path, out):
    rows = [r for r in csv.reader(l for l in open(path) if l.startswith('"'))]
    hdr = rows[0]
    ki, vi, ui = hdr.index("Kernel Name"), hdr.index("Metric Value"), hdr.index("Metric Unit")
    agg = collections.OrderedDict()
    for r in rows[1:]:
        agg.setdefault(r[ki].split("(")[0], []).append(float(r[vi].replace(",", "")))
    tot = sum(sum(v) for v in agg.values())
    with open(out, "w") as f:
        f.write(f"# ncu --metrics gpu__time_duration.sum --clock-control none  ({path}); unit {rows[1][ui]}\n")
        f.write("# cold-cache, serialised launches: compare SHARES, not absolutes\n")
        f.write(f"{'kernel':70s} {'n':>5s} {'mean':>12s} {'total':>14s} {'share':>7s}\n")
        for n, v in agg.items():
            f.write(f"{n[:70]:70s} {len(v):5d} {sum(v) / len(v):12.1f} {sum(v):14.1f} {sum(v) / tot:7.3f}\n")
    print(open(out).read())


def full(rep, out, k3_json=None, k3_pattern="k_window"):
    raw = subprocess.run(["ncu", "-i", rep, "--page", "raw", "--csv"], capture_output=True, text=True).stdout
    rows = list(csv.reader(raw.splitlines()))
    hdr, units = rows[0], rows[1]
    ni = hdr.index("Kernel Name")
    with open(out, "w") as f:
        f.write(f"# ncu --set full --clock-control none --import-source on  ({rep})\n")
        traffic = []
        for r in rows[2:]:
            f.write(f"\n== {r[ni][:100]}\n")
            for k in KEYS:
                if k in hdr:
                    i = hdr.index(k)
                    f.write(f"  {k:72s} {r[i]:>16s} {units[i]}\n")
            if k3_pattern in r[ni] and "dram__bytes_read.sum" in hdr:
                def b(k):
                    i = hdr.index(k)
                    v = float(r[i].replace(",", ""))
                    u = units[i].lower()
                    return v * {"byte": 1, "kbyte": 1e3, "mbyte": 1e6, "gbyte": 1e9}[u]
                traffic.append(b("dram__bytes_read.sum") + b("dram__bytes_write.sum"))
    if k3_json and traffic:
        json.dump({"kernel": k3_pattern, "dram_bytes_per_launch": sum(traffic) / len(traffic), "launches": len(traffic),
                   "source": rep}, open(k3_json, "w"))
    print(open(out).read())


if __name__ == "__main__":
    if sys.argv[1] == "launches":
        launches(sys.argv[2], sys.argv[3])
    else:
        full(*sys.argv[2:])
