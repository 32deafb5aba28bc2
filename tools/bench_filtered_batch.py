"""Batched search with a payload filter per query (rbod_search_masks) against the ways to get the same answers
without it: one shared mask, no filter, and a loop of single-query rbod_search calls.  Prints one JSON line.

Workload: a seeded 10M x 768 bf16 cosine gallery (generated on the GPU), Q = 10 000 seeded queries, k = 10 and 100.
Rows are split into M seeded classes; a class mask allows the rows of one class.  Masks and mask ids are device
tensors (a caller that reuses its masks keeps them there).  Per case: K3 time (CUDA events around the tensor-core
launches, option time_k3), whole-call time (host clock around a call that ends in a stream synchronisation), and
queries/s.  The old way (one rbod_search per filtered request) is timed on the first 200 queries and extrapolated.

Client path: QdrantClient.search_batch(requests=...) with 1 000 requests over 64 class filters on a 1M-row
collection; filter compilation (host) and the device search are timed separately.

Exactness: for 64 sampled queries, the per-query-mask result must equal one rbod_search with that query's mask bit
for bit (ids, fp32 and fp64 scores); a mismatch fails the script.

    python tools/bench_filtered_batch.py [--rows N] [--queries Q] [--repeats R] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
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


def class_masks(labels, M, n):
    import torch

    words = (n + 31) // 32
    out = np.zeros((M, words), dtype=np.uint32)
    bits = np.zeros(words * 32, dtype=np.uint8)
    for c in range(M):
        bits[:n] = labels == c
        out[c] = np.packbits(bits, bitorder="little").view(np.uint32)
    return torch.from_numpy(out.view(np.int32)).cuda()


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--dim", type=int, default=768)
    ap.add_argument("--queries", type=int, default=10_000)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--loop-queries", type=int, default=200)
    ap.add_argument("--client-rows", type=int, default=1_000_000)
    ap.add_argument("--out", default="")
    a = ap.parse_args()

    import torch

    if not torch.cuda.is_available():
        sys.exit("bench_filtered_batch: no CUDA device (this measures the B200 path only)")
    from retrieval_based_object_detection_b200 import Gallery

    n, dim, Q = a.rows, a.dim, a.queries
    result = {"tool": "bench_filtered_batch", **gpu_info(), "rows": n, "dim": dim, "dtype": "bf16", "queries": Q,
              "cases": []}
    gen = torch.Generator("cuda").manual_seed(1234)
    g = Gallery(dim, dtype="bf16", capacity=n)
    for r0 in range(0, n, 1_000_000):
        g.upsert(torch.randn(min(1_000_000, n - r0), dim, device="cuda", generator=gen))
    g.set_option("time_k3", 1)
    queries = torch.randn(Q, dim, device="cuda", generator=gen)
    rng = np.random.default_rng(7)
    half = rng.random(n) < 0.5
    shared = class_masks(half.astype(np.int64) - 1, 1, n)            # class 0 = the allowed half: a 50 % mask
    masks = {M: class_masks(rng.integers(0, M, n), M, n) for M in (16, 256)}
    ids = {M: torch.from_numpy(rng.integers(0, M, Q).astype(np.int32)).cuda() for M in (16, 256)}
    mix = ids[16].clone()
    mix[torch.from_numpy(rng.random(Q) < 0.25).cuda()] = -1

    def timed(label, k, **kw):
        g.search(queries, k, **kw)                                    # warm-up: module load, workspaces
        k3, call = [], []
        for _ in range(a.repeats):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res = g.search(queries, k, **kw)
            torch.cuda.synchronize()
            call.append((time.perf_counter() - t0) * 1e3)
            k3.append(res.stats["k3_ms"])
        c = {"case": label, "k": k, "k3_ms": float(np.median(k3)), "call_ms": float(np.median(call)),
             "qps": Q / (float(np.median(call)) * 1e-3), "k3_ms_all": k3, "call_ms_all": call,
             "fallback_queries": int(res.stats["fallback_queries"]), "sweep_queries": int(res.stats["sweep_queries"])}
        result["cases"].append(c)
        print(json.dumps(c), file=sys.stderr, flush=True)
        return res

    for k in (10, 100):
        timed("no_filter", k)
        timed("shared_mask_50pct", k, row_mask=shared[0])
        timed("per_query_M16", k, row_mask=masks[16], mask_of_query=ids[16])
        timed("per_query_M256", k, row_mask=masks[256], mask_of_query=ids[256])
        timed("per_query_M16_25pct_unfiltered", k, row_mask=masks[16], mask_of_query=mix)
        # the old way: one single-query rbod_search per filtered request
        m256, i256 = masks[256], ids[256].cpu().numpy()
        L = a.loop_queries
        g.search(queries[:1], k, row_mask=m256[int(i256[0])])
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for i in range(L):
            g.search(queries[i:i + 1], k, row_mask=m256[int(i256[i])])
        torch.cuda.synchronize()
        per_q = (time.perf_counter() - t0) / L
        c = {"case": "loop_of_single_query_searches_M256", "k": k, "measured_queries": L,
             "call_ms_per_query": per_q * 1e3, "qps": 1.0 / per_q, "extrapolated_call_ms_for_all_queries": per_q * Q * 1e3,
             "extrapolated": True}
        result["cases"].append(c)
        print(json.dumps(c), file=sys.stderr, flush=True)
        # exactness: 64 sampled queries against one rbod_search each with the query's own mask
        ref = g.search(queries, k, row_mask=m256, mask_of_query=ids[256], want_scores64=True)
        bad = 0
        for i in rng.choice(Q, 64, replace=False):
            one = g.search(queries[i:i + 1], k, row_mask=m256[int(i256[i])], want_scores64=True)
            same = (torch.equal(one.rows[0], ref.rows[i]) and torch.equal(one.scores[0], ref.scores[i])
                    and torch.equal(one.scores64[0], ref.scores64[i]))
            bad += not same
        result[f"bitwise_mismatches_k{k}"] = bad
        if bad:
            print(json.dumps(result))
            sys.exit(f"bench_filtered_batch: {bad} of 64 sampled queries differ from their single-query search (k={k})")
    g.close()
    del masks, shared
    torch.cuda.empty_cache()

    # client path, on an in-memory store: nothing is written to disk
    os.environ["RBOD_GALLERY_DTYPE"] = "bf16"
    from qdrant_client import QdrantClient, models

    c = QdrantClient(location=":memory:")
    nc, M = a.client_rows, 64
    c.recreate_collection("b", vectors_config=models.VectorParams(size=dim, distance=models.Distance.COSINE))
    labels = rng.integers(0, M, nc)
    col = c._root.get("b")
    vec = torch.randn(nc, dim, device="cuda", generator=gen)
    col.upsert_device(list(range(nc)), vec, [{"class_name": f"c{int(x)}"} for x in labels])
    flts = [models.Filter(must=[models.FieldCondition(key="class_name", match=models.MatchValue(value=f"c{j}"))])
            for j in range(M)]
    qv = torch.randn(1000, dim, device="cuda", generator=gen).cpu().numpy()
    reqs = [models.SearchRequest(vector=qv[i].tolist(), filter=flts[int(rng.integers(0, M))], limit=10)
            for i in range(1000)]
    c.search_batch("b", requests=reqs[:10])                       # warm-up
    col._columns_n = -1                                           # the dictionary-encoded column is built again
    t0 = time.perf_counter()
    for f in flts:
        col.filter_mask(f)
    compile_ms = (time.perf_counter() - t0) * 1e3
    dev_ms = []
    orig = col.gallery.search

    def timed_search(*args, **kw):
        torch.cuda.synchronize()
        t = time.perf_counter()
        r = orig(*args, **kw)
        torch.cuda.synchronize()
        dev_ms.append((time.perf_counter() - t) * 1e3)
        return r

    col.gallery.search = timed_search
    t0 = time.perf_counter()
    got = c.search_batch("b", requests=reqs)
    total_ms = (time.perf_counter() - t0) * 1e3
    col.gallery.search = orig
    assert len(got) == 1000 and all(len(p) == 10 for p in got)
    cc = {"case": "client_search_batch_requests", "rows": nc, "requests": 1000, "filters": M, "k": 10,
          "filter_compile_ms_64_filters": compile_ms, "device_search_ms": sum(dev_ms), "device_searches": len(dev_ms),
          "total_ms": total_ms, "requests_per_s": 1000 / (total_ms * 1e-3)}
    result["cases"].append(cc)
    print(json.dumps(cc), file=sys.stderr, flush=True)
    c.close()
    line = json.dumps(result)
    print(line)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
