#!/usr/bin/env python
"""Condenses what a GPU pass left in gpurun_out/ (scratch) into profiles/ (tracked):

    python tools/make_profiles.py r01

* <tag>_launches_bench.csv        -> profiles/<tag>_launches_bench_summary.txt (+ the raw csv)
* <tag>_{k1,k2,k3,...}_full.ncu-rep -> profiles/<tag>_<kernel>_ncu.txt (tracked metrics + hottest SASS lines)
* the K3 capture taken on the bench command -> profiles/k3_traffic.json (read by bench.py for roofline.traffic)
"""
import collections
import csv
import glob
import json
import os
import shutil
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "gpurun_out")
PROF = os.path.join(ROOT, "profiles")


def launches(tag):
    src = os.path.join(OUT, f"{tag}_launches_bench.csv")
    if not os.path.exists(src):
        return
    rows = list(csv.reader(open(src)))
    start = next(i for i, r in enumerate(rows) if r and r[0] == "ID")
    hdr = rows[start]
    ki, vi, ui = hdr.index("Kernel Name"), hdr.index("Metric Value"), hdr.index("Metric Unit")
    tot = collections.OrderedDict()
    for r in rows[start + 1:]:
        if len(r) <= vi:
            continue
        v = float(r[vi].replace(",", "")) * {"ns": 1e-6, "us": 1e-3, "ms": 1.0, "s": 1e3}[r[ui]]
        name = r[ki].split("(")[0].replace("void ", "").replace("rbod::<unnamed>::", "")[-70:]
        a = tot.setdefault(name, [0, 0.0])
        a[0] += 1
        a[1] += v
    mine = ("k3_cosine", "rescore", "merge_partials", "prep_queries", "select_", "tau_init", "l2norm", "seg_", "gather_",
            "merge_topk", "dist_")
    ours = {k: v for k, v in tot.items() if any(m in k for m in mine)}
    total, total_search = sum(v for _, v in tot.values()), sum(v for k, (_, v) in ours.items() if "l2norm" not in k)
    with open(os.path.join(PROF, f"{tag}_launches_bench_summary.txt"), "w") as f:
        f.write("# ncu --metrics gpu__time_duration.sum --clock-control none, command: python bench.py --steps 2 --warmup 3 "
                "--no-cpu-baseline --no-parity\n# cold-cache, serialised launches: compare SHARES, not absolutes\n")
        f.write(f"# total {total:.3f} ms over {sum(n for n, _ in tot.values())} launches; search kernels only "
                f"{total_search:.3f} ms\n")
        for k, (n, v) in sorted(tot.items(), key=lambda x: -x[1][1]):
            share = f"{100 * v / total_search:6.2f}% of search" if k in ours and "l2norm" not in k else " " * 17
            f.write(f"{v:10.3f} ms  x{n:4d}  avg {v / n:9.4f} ms  {share}  {k}\n")
    shutil.copy(src, os.path.join(PROF, f"{tag}_launches_bench.csv"))
    print("wrote launches summary")


def ncu_reports(tag):
    for rep in sorted(glob.glob(os.path.join(OUT, f"{tag}_*_full.ncu-rep"))):
        name = os.path.basename(rep).replace("_full.ncu-rep", "")
        txt = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "ncu_summary.py"), rep, "30"],
                             capture_output=True, text=True).stdout
        with open(os.path.join(PROF, f"{name}_ncu.txt"), "w") as f:
            f.write(f"# ncu --set full --clock-control none --import-source on; report {os.path.basename(rep)}\n")
            f.write(txt)
        print("wrote", name)
        if name.endswith("k3bench"):
            raw = subprocess.run(["ncu", "-i", rep, "--page", "raw", "--csv"], capture_output=True, text=True).stdout
            rows = list(csv.reader(raw.splitlines()))
            hdr, units, vals = rows[0], rows[1], rows[2]
            def get(m):
                v, u = float(vals[hdr.index(m)].replace(",", "")), units[hdr.index(m)]
                return v * {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}[u]
            rd, wr = get("dram__bytes_read.sum"), get("dram__bytes_write.sum")
            json.dump({"rows_per_gpu": 10_000_000, "queries": 10_000, "dim": 768, "k": 10,   # bench.py defaults
                       "dram_bytes_per_launch": rd + wr, "dram_bytes_read": rd, "dram_bytes_write": wr,
                       "source": os.path.basename(rep), "command": "python bench.py --steps 1 --warmup 3 --no-cpu-baseline",
                       "tensor_pipe_active_pct": float(vals[hdr.index("sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_elapsed")])},
                      open(os.path.join(PROF, "k3_traffic.json"), "w"), indent=1)
            print("wrote k3_traffic.json")


if __name__ == "__main__":
    tag = sys.argv[1] if len(sys.argv) > 1 else "r01"
    os.makedirs(PROF, exist_ok=True)
    launches(tag)
    ncu_reports(tag)
