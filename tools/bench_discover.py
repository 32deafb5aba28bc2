"""Discovery and context search throughput (rbod_discover, kernel K7, exact fp64 sweep).  Prints one JSON line.

Galleries (seeded, generated on the GPU): 1M x 512 f32 and 10M x 768 bf16, COSINE.  Workloads, k = 10, no filter, every
example a stored id (its stored row is the example):
  * discovery: 256 requests, each a target and 2 pairs (5 slots; 6 requests = 30 slots a pass);
  * context:   256 requests, each 3 pairs (6 slots; 5 requests = 30 slots a pass).
Timed at the Gallery level (host clock around a call that ends in a stream synchronisation, median of --repeats after a
warm-up).  Per case and workload: requests/s, ms per pass, passes, re-sweeps (requests whose list overflowed and was
tightened), and the achieved fp64 rate 2 * rows * dim * slots / time against the nominal ~37 TFLOP/s fp64 DESIGN.md §3
uses for K5.  The -Xptxas -v figures of the eight K7 instantiations are read from the build's k7_discover.ptxas.log.

Exactness: on the 1M-row gallery, 32 sampled requests of each workload are checked against the fp64 numpy oracle
(oracle/oracle_discover.py ``discover_score``, compared by oracle/oracle_reco.py ``agrees``: scores within rtol 1e-12,
ids equal except among rows the oracle scores within 1e-12 of each other); on both galleries, 32 sampled requests of each workload must equal the same request
sent alone bit for bit.  A mismatch fails the script.

    python tools/bench_discover.py [--repeats R] [--out FILE] [--small]
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
    log = os.path.join(ROOT, "retrieval_based_object_detection_b200", "csrc", "k7_discover.ptxas.log")
    if not os.path.exists(log):
        return []
    text = open(log, encoding="utf-8").read()
    out = []
    for m in re.finditer(r"Function properties for (\S*disc_collect_kernelILi(\d)ELi(\d+)E\S*)\n.*?(\d+) bytes spill stores, "
                         r"(\d+) bytes spill loads.*?Used (\d+) registers", text, flags=re.S):
        out.append({"metric": int(m.group(2)), "ns": int(m.group(3)), "registers": int(m.group(6)),
                    "spill_stores": int(m.group(4)), "spill_loads": int(m.group(5))})
    return out


WORKLOADS = {"discovery": [0, 1, -1, 1, -1], "context": [1, -1, 1, -1, 1, -1]}


def run_case(G, n, dim, dtype, repeats, oracle_check, rng):
    import torch

    from oracle import oracle_np as O
    from oracle import oracle_discover as OD
    from oracle import oracle_reco as OR

    gen = torch.Generator("cuda").manual_seed(4321)
    g = G(dim, dtype=dtype, metric="cosine", capacity=n)
    for r0 in range(0, n, 1_000_000):
        g.upsert(torch.randn(min(1_000_000, n - r0), dim, device="cuda", generator=gen))
    R, k = 256, 10
    stored = g.get_rows(np.arange(n)) if oracle_check else None
    case = {"rows": n, "dim": dim, "dtype": dtype, "metric": "cosine", "requests": R, "k": k, "workloads": {}}
    for name, rl in WORKLOADS.items():
        m = len(rl)
        ids = rng.integers(0, n, (R, m))
        ex = g.get_rows(ids.reshape(-1))                      # the stored rows of the example ids, [m R, dim]
        roles = np.tile(np.array(rl, np.int8), R)
        offsets = np.arange(R + 1, dtype=np.int64) * m
        g.discover(ex, roles, offsets, k)
        ts = []
        for _ in range(repeats):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res = g.discover(ex, roles, offsets, k, want_keys=True)
            torch.cuda.synchronize()
            ts.append(time.perf_counter() - t0)
        t = float(np.median(ts))
        per_pass = 32 // m
        passes = (R + per_pass - 1) // per_pass
        w = {"slots_per_request": m, "requests_per_pass": per_pass, "passes": passes, "requests_per_s": R / t,
             "call_ms": t * 1e3, "call_ms_all": [x * 1e3 for x in ts], "ms_per_pass": t * 1e3 / passes,
             "launches": int(res.stats["total_launches"]), "resweeps": int(res.stats["fallback_queries"]),
             "achieved_fp64_tflops": 2.0 * n * dim * m * R / t / 1e12}
        w["achieved_share_of_nominal_fp64"] = w["achieved_fp64_tflops"] / NOMINAL_FP64_TFLOPS
        sample = rng.choice(R, 32, replace=False)
        bad = 0
        for r in sample:
            one = g.discover(ex[m * r:m * r + m], roles[:m], [0, m], k, want_keys=True)
            bad += not (np.array_equal(one.rows[0], res.rows[r]) and
                        np.array_equal(one.scores64[0].view(np.uint64), res.scores64[r].view(np.uint64)))
        w["alone_bitwise_mismatches_of_32"] = bad
        if oracle_check:
            sel = np.concatenate([np.arange(m * r, m * r + m) for r in sample])
            sc = OD.discover_score(OR.example_keys(ex[sel], stored, "cosine"), np.tile(np.array(rl, np.int8), 32),
                                   np.arange(33) * m, "cosine")
            bad_o = same_ids = 0
            for j, r in enumerate(sample):
                ws, wi = O.topk_from_scores(sc[j:j + 1], k)
                bad_o += not OR.agrees(res.rows[r], res.scores64[r], sc[j], ws[0], wi[0])
                same_ids += int(np.array_equal(res.rows[r], wi[0]))
            w["oracle_mismatches_of_32"] = bad_o
            w["oracle_identical_ids_of_32"] = same_ids   # the rest differ only inside ties within 1e-12 (OR.agrees)
        case["workloads"][name] = w
    case["nominal_fp64_tflops"] = NOMINAL_FP64_TFLOPS
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
        sys.exit("bench_discover: no CUDA device (this measures the B200 path only)")
    from retrieval_based_object_detection_b200 import Gallery

    rng = np.random.default_rng(17)
    result = {"tool": "bench_discover", **gpu_info(), "ptxas_k7": ptxas_figures(), "cases": []}
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
    if any(w["alone_bitwise_mismatches_of_32"] or w.get("oracle_mismatches_of_32")
           for c in result["cases"] for w in c["workloads"].values()):
        sys.exit("bench_discover: sampled requests differ from the oracle or from the request sent alone")


if __name__ == "__main__":
    main()
