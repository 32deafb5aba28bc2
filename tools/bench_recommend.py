"""Recommendation throughput: best_score (rbod_recommend, kernel K6, exact fp64 sweep) against average_vector (one
search of the composed vector).  Prints one JSON line.

Galleries (seeded, generated on the GPU): 1M x 512 f32 and 10M x 768 bf16, COSINE.  Workload: 256 requests, each 2
positive and 1 negative example ids drawn from the gallery (their stored rows are the examples), k = 10, no filter.
Both strategies are timed at the Gallery level (host clock around a call that ends in a stream synchronisation,
median of --repeats after a warm-up).  256 requests x 3 examples pack into passes of 10 requests (30 slots); per
case: requests/s, ms per pass, passes, and the achieved fp64 rate 2 * rows * dim * 768 slots / time against the
nominal ~37 TFLOP/s fp64 DESIGN.md §3 uses for K5.  The -Xptxas -v figures of the eight K6 instantiations are read
from the build's k6_recommend.ptxas.log.

Exactness: on the 1M-row gallery, 32 sampled requests are checked against the fp64 numpy oracle
(oracle/oracle_reco.py ``agrees``: scores within rtol 1e-12, ids equal except among rows the oracle scores within 1e-12 of
each other -- the two positive examples are stored rows and score s(1) against themselves, give or take an ulp, so
their order is a coin toss between two summation orders); on both galleries, 32 sampled requests must equal the
same request sent alone bit for bit.  A mismatch fails the script.

    python tools/bench_recommend.py [--repeats R] [--out FILE]
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

NOMINAL_FP64_TFLOPS = 37.0


def gpu_info() -> dict:
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, check=True).stdout.strip().splitlines()[0]
    name, power = [s.strip() for s in out.split(",")]
    return {"gpu": name, "power_limit": power}


def ptxas_figures() -> list:
    log = os.path.join(ROOT, "retrieval_based_object_detection_b200", "csrc", "k6_recommend.ptxas.log")
    if not os.path.exists(log):
        return []
    text = open(log, encoding="utf-8").read()
    out = []
    for m in re.finditer(r"Function properties for (\S*reco_collect_kernelILi(\d)ELi(\d+)E\S*)\n.*?(\d+) bytes spill stores, "
                         r"(\d+) bytes spill loads.*?Used (\d+) registers", text, flags=re.S):
        out.append({"metric": int(m.group(2)), "ns": int(m.group(3)), "registers": int(m.group(6)),
                    "spill_stores": int(m.group(4)), "spill_loads": int(m.group(5))})
    return out


def run_case(G, n, dim, dtype, repeats, oracle_check, rng):
    import torch

    from oracle import oracle_np as O
    from oracle import oracle_reco as OR

    gen = torch.Generator("cuda").manual_seed(4321)
    g = G(dim, dtype=dtype, metric="cosine", capacity=n)
    for r0 in range(0, n, 1_000_000):
        g.upsert(torch.randn(min(1_000_000, n - r0), dim, device="cuda", generator=gen))
    R, k = 256, 10
    ids = rng.integers(0, n, (R, 3))
    ex = g.get_rows(ids.reshape(-1))                      # the stored rows of the example ids, [3R, dim]
    signs = np.tile(np.array([1, 1, -1], np.int8), R)
    offsets = np.arange(R + 1, dtype=np.int64) * 3
    ex64 = ex.reshape(R, 3, dim).astype(np.float64)
    avg = (2.0 * ex64[:, :2].mean(axis=1) - ex64[:, 2]).astype(np.float32)

    def timed(fn):
        fn()
        ts = []
        for _ in range(repeats):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res = fn()
            torch.cuda.synchronize()
            ts.append(time.perf_counter() - t0)
        return float(np.median(ts)), ts, res

    t_best, all_best, res = timed(lambda: g.recommend(ex, signs, offsets, k, want_keys=True))
    t_avg, all_avg, _ = timed(lambda: g.search(avg, k))
    passes = (R + 9) // 10
    case = {"rows": n, "dim": dim, "dtype": dtype, "metric": "cosine", "requests": R, "examples_per_request": "2+/1-",
            "k": k, "best_score_requests_per_s": R / t_best, "best_score_call_ms": t_best * 1e3,
            "best_score_call_ms_all": [t * 1e3 for t in all_best], "passes": passes,
            "ms_per_pass": t_best * 1e3 / passes, "launches": int(res.stats["total_launches"]),
            "resweeps": int(res.stats["fallback_queries"]),
            "achieved_fp64_tflops": 2.0 * n * dim * 3 * R / t_best / 1e12, "nominal_fp64_tflops": NOMINAL_FP64_TFLOPS,
            "average_vector_requests_per_s": R / t_avg, "average_vector_call_ms": t_avg * 1e3,
            "average_vector_call_ms_all": [t * 1e3 for t in all_avg]}
    case["achieved_share_of_nominal_fp64"] = case["achieved_fp64_tflops"] / NOMINAL_FP64_TFLOPS
    sample = rng.choice(R, 32, replace=False)
    bad = 0
    for r in sample:
        one = g.recommend(ex[3 * r:3 * r + 3], signs[:3], [0, 3], k, want_keys=True)
        bad += not (np.array_equal(one.rows[0], res.rows[r]) and
                    np.array_equal(one.scores64[0].view(np.uint64), res.scores64[r].view(np.uint64)))
    case["alone_bitwise_mismatches_of_32"] = bad
    if oracle_check:
        stored = g.get_rows(np.arange(n))
        sel = np.concatenate([np.arange(3 * r, 3 * r + 3) for r in sample])
        sc = OR.best_score(OR.example_keys(ex[sel], stored, "cosine"), np.tile(np.array([1, 1, -1], np.int8), 32),
                           np.arange(33) * 3, "cosine")
        bad_o = same_ids = 0
        for j, r in enumerate(sample):
            ws, wi = O.topk_from_scores(sc[j:j + 1], k)
            bad_o += not OR.agrees(res.rows[r], res.scores64[r], sc[j], ws[0], wi[0])
            same_ids += int(np.array_equal(res.rows[r], wi[0]))
        case["oracle_mismatches_of_32"] = bad_o
        case["oracle_identical_ids_of_32"] = same_ids   # the rest differ only inside ties within 1e-12 (OR.agrees)
    g.close()
    torch.cuda.empty_cache()
    return case


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default="")
    ap.add_argument("--small", action="store_true", help="only the 1M x 512 f32 gallery")
    a = ap.parse_args()

    import torch

    if not torch.cuda.is_available():
        sys.exit("bench_recommend: no CUDA device (this measures the B200 path only)")
    from retrieval_based_object_detection_b200 import Gallery

    rng = np.random.default_rng(17)
    result = {"tool": "bench_recommend", **gpu_info(), "ptxas_k6": ptxas_figures(), "cases": []}
    shapes = [(1_000_000, 512, "f32", True)] + ([] if a.small else [(10_000_000, 768, "bf16", False)])
    for n, dim, dtype, oracle_check in shapes:
        c = run_case(Gallery, n, dim, dtype, a.repeats, oracle_check, rng)
        result["cases"].append(c)
        print(json.dumps(c), file=sys.stderr, flush=True)
    line = json.dumps(result)
    print(line)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(line + "\n")
    if any(c["alone_bitwise_mismatches_of_32"] or c.get("oracle_mismatches_of_32") for c in result["cases"]):
        sys.exit("bench_recommend: sampled requests differ from the oracle or from the request sent alone")


if __name__ == "__main__":
    main()
