"""Maximal marginal relevance throughput (rbod_search_mmr: the candidate search, then kernel K8).  Prints one JSON line.

Workloads (seeded galleries generated on the GPU, no filter):
  * 10M x 768 bf16 COSINE, Q = 10^4 queries (stored rows plus noise), limit 10, L = 100 candidates, diversity 0.5.  The
    whole call is timed against rbod_search at k = 100 on the same queries, alternating, two runs each (k = 100 builds
    the fp16 shadow of the bf16 gallery, as any such search does; it is built in the warm-up).
  * the same gallery at Q = 1 (median of 20 calls each);
  * 1M x 512 fp32 COSINE: Q = 10^4 at limit 10, L = 100, and Q = 256 at limit 100, L = 1000 (the candidate search takes
    the fp64 sweep, K5, which scores every row of the gallery for every query in fp64).
K8 alone: the device time of its kernel (mmr_select_kernel) in a torch.profiler trace of one call with device inputs,
taken after the timed runs; K8's fp64 rate is 2 Q (limit - 1) L dim over it.

Exactness: 32 sampled queries of each workload equal the same query sent alone bit for bit, and on the 1M gallery they
pass ``oracle_mmr.mmr_agrees``.  A mismatch fails the script.

    python tools/bench_mmr.py [--out FILE] [--small]
"""
from __future__ import annotations

import argparse
import json
import os
import re
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info() -> dict:
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, check=True).stdout.strip().splitlines()[0]
    name, power = [s.strip() for s in out.split(",")]
    return {"gpu": name, "power_limit": power}


def ptxas_figures() -> list:
    log = os.path.join(ROOT, "retrieval_based_object_detection_b200", "csrc", "k8_mmr.ptxas.log")
    if not os.path.exists(log):
        return []
    text = open(log, encoding="utf-8").read()
    return [{"metric": int(m.group(2)), "registers": int(m.group(5)), "spill_stores": int(m.group(3)),
             "spill_loads": int(m.group(4))}
            for m in re.finditer(r"Function properties for (\S*mmr_select_kernelILi(\d)E\S*)\n.*?(\d+) bytes spill "
                                 r"stores, (\d+) bytes spill loads.*?Used (\d+) registers", text, flags=re.S)]


def timed(fn):
    import torch

    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def kernel_ms(fn, name: str) -> float:
    """Device time (ms) of the kernels whose name contains ``name`` in a torch.profiler trace of fn()."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    us = 0.0
    for e in prof.events():
        if name in e.name:
            us += getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
    return us / 1e3


def workload(g, q, limit, L, dim, stored=None, metric="cosine", repeats=2):
    """Whole call vs rbod_search at k = L, alternating; K8 alone from a profiler trace; sampled checks."""
    from oracle import oracle_mmr as OM

    Q = len(q)
    import torch

    g.search_mmr(q, limit, L, 0.5)
    g.search(q, L)
    t_mmr, t_search = [], []
    for _ in range(repeats):
        t, res = timed(lambda: g.search_mmr(q, limit, L, 0.5, want_keys=True))
        t_mmr.append(t)
        t, _ = timed(lambda: g.search(q, L))
        t_search.append(t)
    qd = torch.from_numpy(q).cuda()
    k8_ms = kernel_ms(lambda: g.search_mmr(qd, limit, L, 0.5), "mmr_select")
    w = {"Q": Q, "limit": limit, "candidates": L, "diversity": 0.5,
         "mmr_call_ms": [t * 1e3 for t in t_mmr], "search_call_ms": [t * 1e3 for t in t_search],
         "mmr_over_search": float(np.median(t_mmr) / np.median(t_search)),
         "k8_kernel_ms": k8_ms, "k8_share_of_call": k8_ms / (float(np.median(t_mmr)) * 1e3),
         "k8_fp64_flop": 2.0 * Q * (limit - 1) * L * dim,
         "queries_per_s": Q / float(np.median(t_mmr)), "launches": int(res.stats["total_launches"])}
    w["k8_fp64_tflops"] = w["k8_fp64_flop"] / (k8_ms * 1e-3) / 1e12 if k8_ms > 0 else None
    rng = np.random.default_rng(3)
    sample = rng.choice(Q, min(32, Q), replace=False)
    bad = bad_o = 0
    if stored is not None:
        from oracle import oracle_reco as OR

        qkeys = dict(zip(sample, OR.example_keys(q[sample], stored, metric)))   # one pass over the gallery
    for i in sample:
        one = g.search_mmr(q[i:i + 1], limit, L, 0.5, want_keys=True)
        bad += not (np.array_equal(one.rows[0], res.rows[i]) and
                    np.array_equal(one.scores64[0].view(np.uint64), res.scores64[i].view(np.uint64)))
        if stored is not None:
            prep = OM.prepare(q[i], stored, L, metric, qkeys=qkeys[i])
            bad_o += not OM.mmr_agrees(res.rows[i], q[i], stored, limit, L, 0.5, metric, prepared=prep)
    w["alone_bitwise_mismatches"] = int(bad)
    w["sampled"] = int(len(sample))
    if stored is not None:
        w["oracle_mismatches"] = int(bad_o)
    return w


def make(G, n, dim, dtype, seed):
    import torch

    gen = torch.Generator("cuda").manual_seed(seed)
    g = G(dim, dtype=dtype, metric="cosine", capacity=n)
    for r0 in range(0, n, 1_000_000):
        g.upsert(torch.randn(min(1_000_000, n - r0), dim, device="cuda", generator=gen))
    return g


def queries(g, n, Q, dim, seed):
    rng = np.random.default_rng(seed)
    base = np.asarray(g.get_rows(rng.integers(0, n, Q)))
    return (base + 0.05 * rng.standard_normal((Q, dim))).astype(np.float32)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--small", action="store_true", help="only the 1M x 512 fp32 gallery")
    a = ap.parse_args()

    import torch

    if not torch.cuda.is_available():
        sys.exit("bench_mmr: no CUDA device (this measures the B200 path only)")
    from retrieval_based_object_detection_b200 import Gallery

    result = {"tool": "bench_mmr", **gpu_info(), "ptxas_k8": ptxas_figures(), "cases": []}
    n, dim = 1_000_000, 512
    g = make(Gallery, n, dim, "f32", 11)
    stored = np.asarray(g.get_rows(np.arange(n)))
    q = queries(g, n, 10_000, dim, 12)
    case = {"rows": n, "dim": dim, "dtype": "f32", "metric": "cosine", "workloads": []}
    for limit, L, nq in ((10, 100, 10_000), (100, 1000, 256)):   # L = 1000: every query swept exactly (K5)
        case["workloads"].append(workload(g, q[:nq], limit, L, dim, stored))
        print(json.dumps(case["workloads"][-1]), file=sys.stderr, flush=True)
    result["cases"].append(case)
    g.close()
    del stored
    torch.cuda.empty_cache()
    if not a.small:
        n, dim = 10_000_000, 768
        g = make(Gallery, n, dim, "bf16", 21)
        q = queries(g, n, 10_000, dim, 22)
        case = {"rows": n, "dim": dim, "dtype": "bf16", "metric": "cosine", "workloads": []}
        case["workloads"].append(workload(g, q, 10, 100, dim))
        print(json.dumps(case["workloads"][-1]), file=sys.stderr, flush=True)
        one = q[:1]
        t_m = [timed(lambda: g.search_mmr(one, 10, 100, 0.5))[0] for _ in range(20)]
        t_s = [timed(lambda: g.search(one, 100))[0] for _ in range(20)]
        case["q1"] = {"mmr_call_ms_median": float(np.median(t_m)) * 1e3, "search_call_ms_median": float(np.median(t_s)) * 1e3}
        result["cases"].append(case)
        g.close()
    line = json.dumps(result)
    print(line)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(line + "\n")
    if any(w["alone_bitwise_mismatches"] or w.get("oracle_mismatches") for c in result["cases"] for w in c["workloads"]):
        sys.exit("bench_mmr: sampled queries differ from the oracle or from the query sent alone")


if __name__ == "__main__":
    main()
