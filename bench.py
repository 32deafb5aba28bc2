#!/usr/bin/env python
"""Headline benchmark: top-10 cosine queries/s on a 10M x 768 bf16 gallery (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--rows R --queries Q --k K]
                    [--dump-outputs DIR]

A step = one pass of the hot path over one batch of synthetic queries: rbod_search (query prep,
K3 tcgen05 cosine top-k, merge + fp64 rescoring + certification in the finish kernel) on a gallery
that is already resident in HBM.  ``value`` times the step with device-resident queries/outputs;
``e2e`` times the same call through the C ABI with HOST (pinned) query and result buffers, copies
inside the timed region.  ``roofline`` describes the dominant kernel (K3), timed live with CUDA
events on its launch stream.  ``cpu_baseline`` is the numpy float64 oracle port on a bounded sample
of the same workload (the one place besides tests/smoke where oracle/ is executed; it is never the
thing shipped).  Gallery and queries come from fixed seeds, so ``--dump-outputs`` of two builds run
with the same arguments can be compared array for array.

N > 1 (torchrun, one rank per GPU): the 10M rows are block-partitioned over the ranks, every rank
searches its shard for the same query batch into one packed buffer, ONE NCCL all-gather of the
(2, Q, k) buffers, K4 merge (which also maps local row slots to global ids).  Timing = CUDA events
bracketed by barrier + synchronize, max over ranks.

``configs`` (same JSON line) carries the other BASELINE.json configurations measured at the run's N with their
own parity checks: C4 (top-100 on the same gallery), C2 (1M x 512 fp32, N = 1 only), C3 (delegate build over row
shards + query-vs-centroid top-5) and, at N = 8, C5 (100M x 768 fp16, batch sweep 1..65536).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "top-10 cosine queries/s on 10M x 768"
UNIT = "queries/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--dim", type=int, default=768)
    ap.add_argument("--queries", type=int, default=10_000)
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--dtype", default="bf16")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the float64 exactness check (profiling runs: keeps "
                    "the checker's torch kernels out of the launch list)")
    ap.add_argument("--no-configs", action="store_true", help="skip the side configurations (k=100, C2, C3 with the "
                    "sharded delegate build, the 100M-row sweep at 8 GPUs): profiling runs")
    ap.add_argument("--c5", default="auto", choices=["auto", "on", "off"], help="config C5 (100M x 768 fp16 over the "
                    "ranks, batch sweep): auto = only when the run has 8 GPUs")
    ap.add_argument("--variant", type=int, default=-1, help="override the K3 kernel variant (debug)")
    ap.add_argument("--opt", action="append", default=[], help="library tunable key=value (debug), repeatable")
    ap.add_argument("--sweep", default="", help="comma list of batch sizes: per-size p50 latency and q/s on the "
                    "resident gallery (config C5's query sweep), printed as one JSON line instead of the headline")
    ap.add_argument("--dump-outputs", metavar="DIR", default="", help="after the timed steps, write what the last "
                    "timed step returned as DIR/<name>.npy, so that two builds can be compared output for output")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and (a.impl != "b200" or a.sweep):
        ap.error("--dump-outputs writes the headline search's result: not with --impl reference or --sweep")
    return a


def workload_name(a) -> str:
    return (f"{a.rows / 1e6:g}M x {a.dim} {a.dtype} gallery (synthetic unit-norm rows), "
            f"{a.queries}-query batch, exact top-{a.k} cosine")


DUMP_LIMIT = 64 << 20        # bytes --dump-outputs writes at most


def dump_outputs(path, scores, rows, scores64, limit=DUMP_LIMIT):
    """Writes one search result as path/scores.npy (float32), rows.npy (global row ids, exact in float64) and
    scores64.npy (float64).  A result larger than ``limit`` bytes is cut to a fixed, seeded sample of its queries,
    whose indices go to path/query_index.npy."""
    import numpy as np

    arrays = {"scores": np.asarray(scores, np.float32), "rows": np.asarray(rows, np.float64),
              "scores64": np.asarray(scores64, np.float64)}
    Q = arrays["scores"].shape[0]
    bytes_per_query = sum(x.itemsize * x.shape[1] for x in arrays.values()) + 8        # + its index when sampled
    keep = (limit - 4096) // bytes_per_query                                           # 4096: the .npy headers
    if Q > keep:
        idx = np.sort(np.random.default_rng(0).choice(Q, keep, replace=False))
        arrays = {name: x[idx] for name, x in arrays.items()}
        arrays["query_index"] = idx.astype(np.float64)
    os.makedirs(path, exist_ok=True)
    for name, x in arrays.items():
        np.save(os.path.join(path, f"{name}.npy"), x)


# --------------------------------------------------------------------------------------------
# clocks: sample nvidia-smi while the timed region runs
# --------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            f = tempfile.NamedTemporaryFile("w", suffix=".csv", delete=False)
            self.path = f.name
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=f,
                                         stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        try:
            for line in open(self.path):
                p = [x.strip() for x in line.split(",")]
                if len(p) < 9:
                    continue
                try:
                    sm.append(float(p[1]))
                    mx.append(float(p[2]))
                except ValueError:
                    continue
                try:
                    pw.append(float(p[3]))
                except ValueError:
                    pass
                for name, val in zip(names, p[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "power_w": statistics.median(pw) if pw else None, "reasons": sorted(reasons)}


# --------------------------------------------------------------------------------------------
# CPU legs (oracle port) -- bounded samples, scaled to the metric's unit
# --------------------------------------------------------------------------------------------
def host_threads() -> dict:
    """Threads the CPU legs can use.  torchrun exports OMP_NUM_THREADS=1 to every rank of a multi-GPU launch, which
    would make the N > 1 reference arm run on one core: the legs lift the BLAS pool back to every core."""
    out = {"os_cpu_count": os.cpu_count() or 1, "omp_num_threads_env": os.environ.get("OMP_NUM_THREADS")}
    try:
        import torch

        out["torch_num_threads"] = torch.get_num_threads()
    except Exception:
        out["torch_num_threads"] = None
    return out


class all_cores:
    """Context manager: numpy's BLAS / OpenMP pools use every host core inside it, whatever the launcher exported."""

    def __enter__(self):
        self.ctx = None
        try:
            from threadpoolctl import threadpool_limits

            self.ctx = threadpool_limits(limits=os.cpu_count() or 1)
            self.ctx.__enter__()
        except Exception:
            self.ctx = None
        return self

    def __exit__(self, *exc):
        if self.ctx is not None:
            self.ctx.__exit__(*exc)
        return False


def blas_threads() -> int:
    try:
        from threadpoolctl import threadpool_info

        n = [p.get("num_threads", 1) for p in threadpool_info() if p.get("user_api") == "blas"]
        return max(n) if n else 1
    except Exception:
        return os.cpu_count() or 1


def cpu_sample_qps(a, budget_s: float = 12.0):
    """B2 (BASELINE.md section 3): times the float64 numpy oracle (cosine_topk: GEMM + (score desc, id asc) top-k) on a
    row sample of the gallery with every host core and scales queries/s linearly to the full row count."""
    from oracle import oracle_np as O

    with all_cores():
        threads = blas_threads()
        n_s = min(a.rows, 200_000)
        g = O.l2_normalize_store(O.synthetic_unit_rows(n_s, a.dim, seed=0), a.dtype if a.dtype != "fp16" else "f16")[0]
        q_probe = O.synthetic_unit_rows(32, a.dim, seed=1)
        t0 = time.perf_counter()
        O.cosine_topk(q_probe, g, a.k)
        t_probe = time.perf_counter() - t0
        q_s = int(max(32, min(a.queries, 32 * budget_s / max(t_probe, 1e-3))))
        q = O.synthetic_unit_rows(q_s, a.dim, seed=2)
        t0 = time.perf_counter()
        O.cosine_topk(q, g, a.k)
        t = time.perf_counter() - t0
    qps_full = q_s / t * (n_s / a.rows)
    sample = (f"{q_s} queries x {n_s} rows x {a.dim} (float64 GEMM + partition/lexsort top-{a.k}) in {t:.2f} s; "
              f"queries/s scaled by {n_s}/{a.rows} rows")
    return qps_full, threads, sample, t


def reference_literal_legs(a) -> dict:
    """B1 and B3 of BASELINE.md section 3 -- the reference's own two functions on this path, run the way its scripts
    run them (one Python call per pair / per class, one core).  With /root/reference present the functions are the
    reference's own objects (AST-extracted cosine_similarity, imported compute_average); on the GPU box, where the
    reference tree does not exist, they are the oracle's line-by-line restatements of 33_...py:76-77 and 32_...py:9-10,
    which tests/test_oracle_golden.py pins bit-for-bit against the originals."""
    import numpy as np

    from oracle import oracle_np as O

    cos, avg, kind = O.cosine_similarity, O.compute_average, "port (oracle restatement; /root/reference absent)"
    try:
        from oracle import ref_loader

        if ref_loader.available():
            cos, avg, kind = ref_loader.cosine_similarity(), ref_loader.delegate_module().compute_average, "reference"
    except Exception:
        pass
    rng = np.random.default_rng(0)
    # B1: 1000 test vectors x 32 delegates, float64 512-d, one cosine_similarity call per pair (33_...py:151)
    tv = rng.standard_normal((1000, 512))
    dv = rng.standard_normal((32, 512))
    t0 = time.perf_counter()
    acc = 0.0
    for i in range(1000):
        for j in range(32):
            acc += cos(tv[i], dv[j])
    t1 = time.perf_counter() - t0
    pairs_s = 32000 / t1
    # B3: compute_average over 10^4 classes x 100 rows x dim (+ the float64 renormalisation Qdrant applies on upsert)
    rows = rng.standard_normal((100 * 200, a.dim)).astype(np.float32)      # 200 distinct classes, cycled 50 times
    t0 = time.perf_counter()
    for c in range(10_000):
        v = np.array(rows[(c % 200) * 100:(c % 200 + 1) * 100], dtype=np.float64)   # np.array([r.vector ...]) 32_...py:137
        m = avg(v)
        m = m / np.linalg.norm(m)
    t3 = time.perf_counter() - t0
    return {"kind": kind, "cores": 1,
            "B1_cosine_similarity_pairs_per_s": pairs_s,
            "B1_sample": f"1000 x 32 pairs, float64 512-d, Python loop, {t1:.2f} s (33_run_all_experiments.py:76-77,151)",
            "B1_queries_per_s_at_full_gallery": pairs_s / a.rows,
            "B3_compute_average_classes_per_s": 10_000 / t3,
            "B3_gbs": 10_000 * 100 * a.dim * 4 / t3 / 1e9,
            "B3_sample": f"10^4 classes x 100 rows x {a.dim}, float64 mean + renormalise per class, {t3:.2f} s "
                         "(32_create_delegate_vector.py:9-10,137)",
            "B4_qdrant_local_mode": "n/a offline (qdrant-client is not installable here)"}


def run_reference(a):
    """--impl reference: the reference's CPU arithmetic for this path (numpy float64 cosine, as
    33_run_all_experiments.py:76-77, batched; the Qdrant server itself is not installable offline),
    on the box's host cores, each step a bounded sample."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    per_step = []
    sample = ""
    threads = os.cpu_count() or 1
    total = a.warmup + a.steps
    budget = max(2.0, min(12.0, 150.0 / max(total, 1)))
    for i in range(total):
        qps, threads, sample, t = cpu_sample_qps(a, budget_s=budget)
        if i >= a.warmup:
            per_step.append((qps, t))
    value = statistics.mean(q for q, _ in per_step)
    ms = statistics.mean(t for _, t in per_step) * 1e3
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(a), "note": "CPU; each step is a bounded row/query sample, scaled"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                         "threads": host_threads()},
        "reference_literal": reference_literal_legs(a),
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# --------------------------------------------------------------------------------------------
# B200 arm
# --------------------------------------------------------------------------------------------
def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return p.get("bf16_tflops_sustained", 1422.9), p.get("bf16_tflops", 1691.8), p.get("hbm_gbs", 6555.8), "measured"
    return 1400.0, 1590.0, 6650.0, "fallback"


class Env:
    """What one rank of the run knows: its place in the process group, its device, the measured peaks."""

    def __init__(self):
        import torch
        import torch.distributed as dist

        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        if self.world > 1:
            # keep stdout to the one JSON line of the contract: NCCL prints its version banner there at the VERSION
            # level, which an nccl.conf on the box can select even when the variable is unset
            if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
                os.environ["NCCL_DEBUG"] = "WARN"
            # a rank that falls out of step must cost minutes, not the default 10-minute watchdog on every GPU
            import datetime

            dist.init_process_group("nccl", device_id=self.dev, timeout=datetime.timedelta(seconds=240))
        self.sus, self.burst, self.hbm, self.peak_src = load_peaks()

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, ms: float) -> float:
        if self.world > 1:
            t = self.torch.tensor([ms], device=self.dev, dtype=self.torch.float64)
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
            return float(t.item())
        return ms

    def timed(self, fn, steps) -> float:
        """Device time of `steps` calls of fn: CUDA events bracketed by barrier + synchronize, max over ranks (ms)."""
        torch = self.torch
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return self.max_over_ranks(e0.elapsed_time(e1))

    def finish(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def build_gallery(E: Env, n_total, dim, dtype, seed, opts=()):
    """This rank's block of a synthetic gallery of n_total unit-norm rows, generated on the device and stored by K1.
    -> (gallery, first global row, local rows, [(event0, event1, rows)] of the K1 launches)."""
    from retrieval_based_object_detection_b200 import Gallery, shard_range

    torch = E.torch
    r0, r1 = shard_range(n_total, E.rank, E.world)
    n_loc = r1 - r0
    gal = Gallery(dim, dtype=dtype, capacity=n_loc, device=E.local_rank)
    gal.set_option("time_k3", 1)
    for kv in opts:                                       # before the first upsert: some options shape the storage
        key, _, val = kv.partition("=")
        gal.set_option(key, int(val))
    gen = torch.Generator(E.dev).manual_seed(seed + E.rank)
    events = []
    for s in range(0, n_loc, 500_000):
        m = min(500_000, n_loc - s)
        x = torch.randn(m, dim, device=E.dev, generator=gen)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        gal.upsert(x)                                     # K1 l2norm_pack: fp32 in, stored rows out
        e1.record()
        events.append((e0, e1, m))
    torch.cuda.synchronize()
    return gal, r0, n_loc, events


class Searcher:
    """One search step: Gallery.search on one GPU, ShardedGallery.search (the public multi-GPU call) on several."""

    def __init__(self, E: Env, gal, Q, k, offs):
        torch = E.torch
        self.E, self.g, self.Q, self.k, self.offs = E, gal, Q, k, offs
        self.packed = torch.empty((2, Q, k), dtype=torch.int64, device=E.dev)          # [0] fp64 scores, [1] local rows
        self.s32 = torch.empty((Q, k), dtype=torch.float32, device=E.dev)
        self.host = (torch.empty((Q, k), dtype=torch.float32).pin_memory(), torch.empty((Q, k), dtype=torch.int64).pin_memory(),
                     torch.empty((Q, k), dtype=torch.float64).pin_memory())
        self.host_np = tuple(t.numpy() for t in self.host)
        self.launches = 0
        self.stats = None
        self.sg = None
        if E.world > 1:                                  # total rows from the shard offsets + the last shard's own count
            cnt = E.torch.tensor([gal.count], dtype=E.torch.int64, device=E.dev)
            E.dist.all_reduce(cnt)
            self.n_total = int(cnt.item())

    def local_out(self):
        return (self.s32, self.packed[1], self.packed[0].view(self.E.torch.float64))

    def shard_view(self):
        if self.sg is None:
            from retrieval_based_object_detection_b200 import ShardedGallery

            self.sg = ShardedGallery.wrap(self.g, self.n_total)
            assert self.sg.shard_offsets() == list(self.offs)
        return self.sg

    def device_step(self, q):
        """queries and results stay on the device -> (scores f32, global ids, scores f64)"""
        if self.E.world == 1:
            res = self.g.search(q, self.k, out=self.local_out())
            self.stats = res.stats
            self.launches += res.stats["total_launches"]
            return self.local_out()
        # the public multi-GPU call (ShardedGallery.search): local search, ONE packed all-gather, K4 merge -- or, from
        # k = 32 on, the split form with the global cut exchanged before the exact rescoring
        sg = self.shard_view()
        out = sg.search(q, self.k)
        self.stats = sg.last_stats
        self.launches += sg.last_stats["total_launches"]        # ours: local search kernels + K4 (NCCL's not counted)
        return out

    def host_step(self, q_np):
        """queries from pinned host memory, (merged) results back into pinned host memory"""
        if self.E.world == 1:
            res = self.g.search(q_np, self.k, out=self.host_np)
            self.launches += res.stats["total_launches"]
            return self.host_np
        # each rank uploads 1/G of the batch over its own PCIe link + an all-gather over NVLink, then as device_step,
        # results into the pinned host buffers, one synchronisation
        sg = self.shard_view()
        sg.search(q_np, self.k, out_host=self.host)
        self.launches += sg.last_stats["total_launches"]        # ours: local search kernels + K4 (NCCL's not counted)
        return self.host_np


def parity_check(E: Env, gal, row0, n_loc, q, k, got, n_check=64):
    """Exactness check outside every timed region: queries against a float64 brute force over the rows as stored
    (torch on the device, row chunks; checker only).  This is the north star's "exact top-k parity" and stands in for
    recall against the reference's Qdrant path, which is not installable offline."""
    torch, dist = E.torch, E.dist
    nq = min(n_check, q.shape[0])
    got_ids, got_s = got[1][:nq].clone(), got[2][:nq].clone()
    qd = q[:nq].double()
    qd = qd / qd.norm(dim=1, keepdim=True)
    best_s = torch.full((nq, 0), 0.0, dtype=torch.float64, device=E.dev)
    best_i = torch.zeros((nq, 0), dtype=torch.int64, device=E.dev)
    step = 250_000
    for s0 in range(0, n_loc, step):
        idx = torch.arange(s0, min(s0 + step, n_loc), device=E.dev)
        rows = gal.get_rows(idx).double()
        sc = (qd @ rows.T) / rows.norm(dim=1)[None, :]
        cs, ci = torch.cat([best_s, sc], 1), torch.cat([best_i, (idx + row0)[None, :].expand(nq, -1)], 1)
        top = torch.topk(cs, min(k, cs.shape[1]), dim=1)
        best_s, best_i = top.values, torch.gather(ci, 1, top.indices)
        del rows, sc, cs, ci
    if E.world > 1:                                      # merge the per-shard exact lists the same way
        gs = torch.empty((E.world,) + tuple(best_s.shape), dtype=best_s.dtype, device=E.dev)
        gi = torch.empty((E.world,) + tuple(best_i.shape), dtype=best_i.dtype, device=E.dev)
        dist.all_gather_into_tensor(gs, best_s.contiguous())
        dist.all_gather_into_tensor(gi, best_i.contiguous())
        cs, ci = gs.permute(1, 0, 2).reshape(nq, -1), gi.permute(1, 0, 2).reshape(nq, -1)
        o = torch.argsort(ci, dim=1, stable=True)        # (score desc, id asc): by id first, then a stable sort by score
        cs, ci = torch.gather(cs, 1, o), torch.gather(ci, 1, o)
        o = torch.argsort(cs, dim=1, descending=True, stable=True)[:, :k]
        best_s, best_i = torch.gather(cs, 1, o), torch.gather(ci, 1, o)
    same = (best_i == got_ids)
    recall = sum(len(set(best_i[i].tolist()) & set(got_ids[i].tolist())) for i in range(nq)) / float(nq * k)
    return {"queries_checked": nq, "ids_identical": bool(same.all().item()), "recall_at_k": recall,
            "max_rel_score_err": float(((best_s - got_s).abs() / best_s.abs().clamp_min(1e-30)).max().item()),
            "against": "float64 brute force over the stored rows (torch, on device); the reference's Qdrant "
                       "path is not installable offline"}


def sweep(E: Env, g, n_local, dim, k, batch_sizes, qgen, offs=None, sharded=False, max_iters=30):
    """Per batch size: p50 / min latency of the whole search (local rbod_search, plus all-gather + K4 when sharded) and
    its fraction of the bound max(bytes / HBM peak, flops / bf16 burst peak) of ONE rank's shard."""
    torch, dist = E.torch, E.dist
    rows_out = []
    for Q in batch_sizes:
        qd = torch.randn(Q, dim, device=E.dev, generator=qgen)
        S = Searcher(E, g, Q, k, offs)
        run = (lambda: S.device_step(qd)) if sharded else (lambda: setattr(S, "stats", g.search(qd, k, out=S.local_out()).stats))
        for _ in range(3):
            run()
        # the iteration count must be the same on every rank (each iteration holds a barrier): derive it from the
        # slowest rank's K3 time, not from this rank's own
        k3_ref = torch.tensor([float(S.stats["k3_ms"])], device=E.dev, dtype=torch.float64)
        if sharded and E.world > 1:
            dist.all_reduce(k3_ref, op=dist.ReduceOp.MAX)
        iters = max(5, min(max_iters, int(2000 / max(1.0, float(k3_ref.item())))))
        lat, k3 = [], []
        for _ in range(iters):
            if sharded:
                E.barrier()
            else:
                torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            run()
            e1.record()
            torch.cuda.synchronize()
            lat.append(e0.elapsed_time(e1))
            k3.append(S.stats["k3_ms"])
        if sharded and E.world > 1:                      # a sharded search is as slow as its slowest rank
            t = torch.tensor(lat, device=E.dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            lat = t.tolist()
        p50 = statistics.median(lat)
        flops, byts = 2.0 * Q * n_local * dim, n_local * dim * 2.0 + Q * dim * 2.0 + Q * k * 12.0
        st = S.stats
        rows_out.append({"Q": Q, "p50_ms": round(p50, 4), "min_ms": round(min(lat), 4), "qps": round(Q / p50 * 1e3, 1),
                         "k3_ms_p50": round(statistics.median(k3), 4),
                         "tflops_per_gpu": round(flops / p50 / 1e9, 1), "gbs_per_gpu": round(byts / p50 / 1e6, 1),
                         "bound": "hbm" if byts / E.hbm / 1e9 > flops / E.burst / 1e12 else "tensor",
                         "frac_of_bound": round(max(byts / E.hbm / 1e9, flops / E.burst / 1e12) / (p50 / 1e3), 3),
                         # back-to-back iterations run at the power-capped clock: the same bound with the SUSTAINED bf16 peak
                         "frac_of_bound_sustained": round(max(byts / E.hbm / 1e9, flops / E.sus / 1e12) / (p50 / 1e3), 3),
                         "slices": st["slices"], "fallback": st["fallback_queries"], "iters": iters})
    return rows_out


def run_b200(a):
    from retrieval_based_object_detection_b200 import shard_range

    E = Env()
    torch, dist = E.torch, E.dist
    world, rank, dev = E.world, E.rank, E.dev
    if world != a.gpus and world > 1:
        raise SystemExit(f"--gpus {a.gpus} but WORLD_SIZE={world}")
    sus, burst, hbm = E.sus, E.burst, E.hbm
    offsets_all = [shard_range(a.rows, r, world)[0] for r in range(world)]

    t_build0 = time.perf_counter()
    g, r0, n_local, k1_events = build_gallery(E, a.rows, a.dim, a.dtype, 1234, a.opt)
    if a.variant >= 0:
        g.set_option("k3_variant", a.variant)
    torch.cuda.synchronize()
    t_build = time.perf_counter() - t_build0

    # ---- the two HBM-bound kernels of the path, measured on the side (not part of the timed step):
    # K1 during the build above (the first chunk is the warm-up), K2 over classes of 100 consecutive rows (4M rows)
    def side_kernels():
        out = []
        esz = 4 if a.dtype in ("f32", "fp32") else 2
        timed_ev = k1_events[1:] or k1_events
        ms = sum(e0.elapsed_time(e1) for e0, e1, _ in timed_ev)
        rows = sum(m for _, _, m in timed_ev)
        out_bytes = 2 + (4 if esz == 4 else 0)            # 16-bit operand (+ fp32 master for fp32 collections)
        gbs = rows * a.dim * (4 + out_bytes) / ms / 1e6
        out.append({"kernel": "l2norm_pack (K1, rbod_upsert)", "bound": "hbm", "achieved": gbs, "peak": hbm,
                    "unit": "GB/s", "frac": gbs / hbm, "algorithmic": f"dim*(4+{out_bytes}) bytes per row, {rows} rows"})
        n2 = min(n_local, 4_000_000)
        C = n2 // 100
        if C >= 1:
            off = torch.arange(0, C * 100 + 1, 100, device=dev, dtype=torch.int64)
            for _ in range(2):
                g.segment_mean(off)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(5):
                g.segment_mean(off)
            e1.record()
            torch.cuda.synchronize()
            ms2 = e0.elapsed_time(e1) / 5
            b2 = C * 100 * a.dim * esz + C * a.dim * 4
            out.append({"kernel": f"segment_mean_renorm (K2, rbod_segment_mean, whole call, {a.dtype} rows)", "bound": "hbm",
                        "achieved": b2 / ms2 / 1e6, "peak": hbm, "unit": "GB/s", "frac": b2 / ms2 / 1e6 / hbm,
                        "algorithmic": f"{C} classes x 100 rows x dim*{esz} bytes + {C}*dim*4 bytes out"})
        return out

    other_kernels = side_kernels()          # every rank (keeps the ranks in step); rank 0's numbers are reported

    qgen = torch.Generator(dev).manual_seed(99)          # same queries on every rank
    q_dev = torch.randn(a.queries, a.dim, device=dev, generator=qgen)
    q_host = torch.empty((a.queries, a.dim), dtype=torch.float32).pin_memory()
    q_host.copy_(q_dev)

    if a.sweep:
        rows_out = sweep(E, g, n_local, a.dim, a.k, [int(x) for x in a.sweep.split(",")], qgen)
        if rank == 0:
            print(json.dumps({"sweep": rows_out, "rows_per_gpu": n_local, "dim": a.dim, "dtype": a.dtype, "k": a.k,
                              "n_gpus": world, "peaks": "measured hbm_gbs / bf16_tflops (burst)"}))
        E.finish()
        return

    S = Searcher(E, g, a.queries, a.k, offsets_all)
    k3_ms, fallback = [], []
    diag = {"search_s": 0.0, "steps": 0, "sweep": 0, "retries": 0}
    last = {}

    def step_device():
        t_s = time.perf_counter()
        out = last["out"] = S.device_step(q_dev)
        diag["search_s"] += time.perf_counter() - t_s
        diag["steps"] += 1
        diag["sweep"] += S.stats["sweep_queries"]
        diag["retries"] += S.stats["presample_retries"]
        k3_ms.append(S.stats["k3_ms"])
        fallback.append(S.stats["fallback_queries"])
        return out

    for _ in range(max(a.warmup, 3)):
        step_device()
    parity = None if a.no_parity else parity_check(E, g, r0, n_local, q_dev, a.k, step_device())
    sampler = ClockSampler(E.local_rank)
    if rank == 0:
        sampler.start()
    S.launches = 0
    k3_ms.clear()
    fallback.clear()
    diag.update(search_s=0.0, steps=0, sweep=0, retries=0)
    ms_dev = E.timed(step_device, a.steps)
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, *(t.cpu().numpy() for t in last["out"]))
    per_rank = {"rank": rank, "search_ms_per_step": round(diag["search_s"] / max(diag["steps"], 1) * 1e3, 3),
                "k3_ms": round(statistics.mean(k3_ms), 3) if k3_ms else 0.0,
                "uncertified_per_step": statistics.mean(fallback) if fallback else 0,
                "sweep_queries": diag["sweep"], "presample_retries": diag["retries"]}
    if world > 1:
        gathered = [None] * world
        dist.all_gather_object(gathered, per_rank)
        per_rank = gathered
    else:
        per_rank = [per_rank]
    n_launch_timed = S.launches
    k3_timed = list(k3_ms)
    last_stats = dict(S.stats)
    for _ in range(2):
        S.host_step(q_host.numpy())
    ms_e2e = E.timed(lambda: S.host_step(q_host.numpy()), a.steps)
    clocks = sampler.stop() if rank == 0 else {}

    configs = [] if a.no_configs else side_configs(a, E, g, r0, n_local, q_dev)

    if rank != 0:
        E.finish()
        return

    value = a.queries * a.steps / (ms_dev / 1e3)
    e2e_value = a.queries * a.steps / (ms_e2e / 1e3)
    k3_avg_ms = statistics.mean(k3_timed) if k3_timed else 0.0
    flops_per_launch = 2.0 * a.queries * n_local * a.dim
    achieved = flops_per_launch / (k3_avg_ms / 1e3) / 1e12 if k3_avg_ms > 0 else 0.0
    roofline = {"bound": "tensor", "kernel": "k3_cosine_topk_kernel", "achieved": achieved, "peak": sus,
                "unit": "TFLOP/s", "frac": achieved / sus, "frac_of_burst": achieved / burst, "traffic": None,
                "peak_source": f"{E.peak_src} bf16_tflops_sustained (kernel timed inside a long step); burst {burst}",
                "algorithmic": f"2*Q*N_local*D = {flops_per_launch:.3e} flop per launch", "kernel_ms": k3_avg_ms,
                "kernel_share_of_step": k3_avg_ms * a.steps / ms_dev if ms_dev > 0 else None}
    # dram bytes per K3 launch from the committed ncu --set full capture -- only when it was taken on this shape
    prof = os.path.join(ROOT, "profiles", "k3_traffic.json")
    if os.path.exists(prof):
        try:
            t = json.load(open(prof))
            if (t.get("rows_per_gpu"), t.get("queries"), t.get("dim"), t.get("k")) == (n_local, a.queries, a.dim, a.k):
                roofline["traffic"] = t.get("dram_bytes_per_launch")
                roofline["traffic_source"] = t.get("source")
        except Exception:
            pass

    cpu = None
    if not a.no_cpu_baseline:
        qps, threads, sample, _ = cpu_sample_qps(a)
        cpu = {"value": qps, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample, "threads": host_threads(),
               "reference_literal": reference_literal_legs(a)}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3),
        "ms_per_step": ms_dev / a.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": a.dtype, "data": "synthetic",
        "config": {"workload": workload_name(a), "gallery_rows_total": a.rows, "rows_per_gpu": n_local, "dim": a.dim,
                   "queries_per_step": a.queries, "k": a.k,
                   "parallelism": f"row-shard x{world} + one packed allgather + K4 merge (top-100: global cut exchanged first)",
                   "l2": "gallery operand per GPU is far larger than the 126 MB L2; no flush between steps",
                   "candidates_per_query": last_stats["candidates"], "slices": last_stats["slices"],
                   "fallback_queries_per_step": statistics.mean(fallback) if fallback else 0,
                   "gallery_build_s": round(t_build, 2), "options": a.opt, "per_rank": per_rank},
        # whole job: the query batch crosses PCIe once (each rank uploads 1/N of it, an all-gather over NVLink completes
        # it on every GPU); every rank reads the merged answer back
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": a.queries * a.dim * 4,
                "d2h_bytes_per_step": world * a.queries * a.k * (4 + 8 + 8), "ms_per_step": ms_e2e / a.steps,
                "call": "Gallery.search" if world == 1 else "ShardedGallery.search(host queries, out_host=pinned buffers)"},
        "gpu_launches": n_launch_timed,
        "roofline": roofline,
        "other_kernels": other_kernels,
        "configs": configs,
        "parity": parity,
        "cpu_baseline": cpu,
        "clocks": clocks,
    }
    print(json.dumps(line))
    E.finish()


def side_configs(a, E: Env, g, r0, n_local, q_dev):
    """The other BASELINE.json configurations at this run's N, each with its own exactness check (every rank runs
    them -- they contain collectives -- rank 0's record is printed)."""
    from retrieval_based_object_detection_b200 import Gallery, ShardedGallery, shard_range

    torch, dist = E.torch, E.dist
    world, rank, dev = E.world, E.rank, E.dev
    sus, burst, hbm = E.sus, E.burst, E.hbm
    out = []
    offsets_all = [shard_range(a.rows, r, world)[0] for r in range(world)]

    def guarded(name, fn):
        try:
            rec = fn()
        except Exception as exc:  # noqa: BLE001 -- a failing side configuration must not take the headline line down
            rec = {"config": name, "error": repr(exc)[:300]}
        if rec is not None:
            out.append(rec)

    # ---- C4: top-100 on the same gallery (BASELINE config 4: 10M x 768 bf16 over 2/4/8 GPUs, allgather merge).  The
    # first k > 40 search makes a bf16 collection build its fp16 search operand (one pass, outside the timing).
    def c4():
        k = 100
        S = Searcher(E, g, a.queries, k, offsets_all)
        k3, fb = [], []

        def step():
            res = S.device_step(q_dev)
            k3.append(S.stats["k3_ms"])
            fb.append(S.stats["fallback_queries"])
            return res

        for _ in range(3):
            step()
        par = parity_check(E, g, r0, n_local, q_dev, k, step())
        k3.clear()
        fb.clear()
        steps = 3
        ms = E.timed(step, steps)
        q_np = q_dev.cpu().numpy()
        for _ in range(2):
            S.host_step(q_np)
        ms_h = E.timed(lambda: S.host_step(q_np), steps)
        k3m = statistics.mean(k3)
        unc = statistics.mean(fb) / a.queries
        tf = 2.0 * a.queries * n_local * a.dim / (k3m / 1e3) / 1e12
        extra = {}
        if world > 1:
            # the same steps with every rank rescoring its own k candidates (no global cut exchanged first)
            sgv = S.shard_view()
            extra["split_search"] = dict(sgv.last_split or {})
            keep_min = sgv.split_min_k
            sgv.split_min_k = 1 << 30
            for _ in range(2):
                step()
            extra["value_without_global_cut"] = a.queries * steps / (E.timed(step, steps) / 1e3)
            sgv.split_min_k = keep_min
        return {"config": "C4: 10M x 768 bf16, top-100, row shards + allgather merge", "k": k, "n_gpus": world, **extra,
                "queries_per_step": a.queries, "value": a.queries * steps / (ms / 1e3), "unit": UNIT,
                "ms_per_step": ms / steps, "e2e_value": a.queries * steps / (ms_h / 1e3), "k3_ms": k3m, "k3_tflops": tf,
                "k3_frac_of_sustained": tf / sus, "uncertified_fraction": unc,
                "candidates": S.stats["candidates"],
                "search_operand": "fp16 shadow of the bf16 rows (built on the first k > 40 search)", "parity": par}

    guarded("C4", c4)

    # ---- C3: delegate vectors over 1M labelled 768-d fp32 rows (10k classes) spread over the ranks, then the
    # query-vs-centroid top-5 search.  The sharded build (per-rank K2 sums + all-reduce + finish) is checked against
    # the single-GPU K2 over all rows, which every rank can afford to hold at this size.
    def c3():
        n, dim, C = 1_000_000, 768, 10_000
        gen = torch.Generator(dev).manual_seed(4321)     # same data on every rank
        labels = torch.randperm(n, device=dev, generator=gen) % C
        full = Gallery(dim, dtype="f32", capacity=n, device=dev.index)
        sg = ShardedGallery(dim, n, dtype="f32", device=dev.index) if world > 1 else None
        a0, a1 = shard_range(n, rank, world)
        for s in range(0, n, 250_000):
            x = torch.randn(250_000, dim, device=dev, generator=gen)
            full.upsert(x)
            if sg is not None:
                lo, hi = max(s, a0), min(s + 250_000, a1)
                if hi > lo:
                    sg.upsert_local(x[lo - s:hi - s])
        order = torch.argsort(labels, stable=True)
        off = torch.zeros(C + 1, dtype=torch.int64, device=dev)
        off[1:] = torch.cumsum(torch.bincount(labels, minlength=C), 0)
        want = full.segment_mean(off, row_idx=order)
        for _ in range(2):
            full.segment_mean(off, row_idx=order)
        ms1 = E.timed(lambda: full.segment_mean(off, row_idx=order), 5) / 5
        alg = n * dim * 4 + n * 8 + C * dim * 4
        rec = {"config": "C3: delegate vectors, 1M x 768 fp32 rows, 10k classes, then query-vs-centroid top-5",
               "n_gpus": world, "k2_single_gpu_ms": ms1, "k2_single_gpu_gbs": alg / ms1 / 1e6,
               "k2_single_gpu_frac_of_hbm": alg / ms1 / 1e6 / hbm,
               "algorithmic_bytes": "n*dim*4 (rows) + n*8 (row index) + C*dim*4 (out)"}
        if sg is not None:
            lab_loc = labels[a0:a1]
            order_loc = torch.argsort(lab_loc, stable=True)
            off_loc = torch.zeros(C + 1, dtype=torch.int64, device=dev)
            off_loc[1:] = torch.cumsum(torch.bincount(lab_loc, minlength=C), 0)
            got = sg.segment_mean(off_loc, row_idx=order_loc)
            ulp = (got.view(torch.int32).long() - want.view(torch.int32).long()).abs().max()
            t = torch.tensor([float(ulp)], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            for _ in range(2):
                sg.segment_mean(off_loc, row_idx=order_loc)
            msN = E.timed(lambda: sg.segment_mean(off_loc, row_idx=order_loc), 5) / 5
            rec.update({"k2_sharded_ms": msN, "k2_sharded_gbs_aggregate": alg / msN / 1e6,
                        "k2_sharded_frac_of_hbm_x_gpus": alg / msN / 1e6 / (hbm * world),
                        "k2_sharded_max_ulp_vs_single_gpu": float(t.item()), "ok": bool(t.item() <= 1.0),
                        "collectives": "all-reduce of [C, dim] fp64 sums (61 MB) + [C] counts per build"})
            sg.local.close()
        # the other three delegate types of 32_create_delegate_vector.py:12-26 on the same classes (K2b, one CTA per class,
        # fp64 like the reference): centroid / weighted re-read the class 2-3 times (L2 hits), the medoid is O(n^2 d)
        k2b = {}
        for kind in ("centroid", "weighted", "medoid"):
            full.segment_delegates(kind, off, row_idx=order)
            ms_k = E.timed(lambda: full.segment_delegates(kind, off, row_idx=order), 3) / 3
            k2b[kind] = {"ms": ms_k, "gbs": alg / ms_k / 1e6, "frac_of_hbm": alg / ms_k / 1e6 / hbm}
        n_c = n // C
        nb = (n_c + 3) // 4
        pairs = nb * (nb + 1) // 2 * 16                  # the tiled kernel computes 4x4 blocks of the upper triangle only
        k2b["medoid"]["fp64_tflops"] = 3.0 * C * pairs * dim / (k2b["medoid"]["ms"] / 1e3) / 1e12
        k2b["medoid"]["bound"] = ("fp64 CUDA cores: 3 flop (DADD, DFMA) per (member pair of the upper triangle, column); no "
                                  "measured fp64 peak on this pool (nominal B200 fp64: ~37 TFLOP/s)")
        rec["k2b_other_delegates"] = k2b
        # query-vs-centroid top-5: 10^4 queries against the 10^4 delegates
        cent = Gallery(dim, dtype="f32", capacity=C, device=dev.index)
        cent.upsert(want)
        q = torch.randn(10_000, dim, device=dev, generator=gen)
        o3 = (torch.empty((10_000, 5), dtype=torch.float32, device=dev), torch.empty((10_000, 5), dtype=torch.int64, device=dev),
              torch.empty((10_000, 5), dtype=torch.float64, device=dev))
        for _ in range(3):
            cent.search(q, 5, out=o3)
        ms_c = E.timed(lambda: cent.search(q, 5, out=o3), 10) / 10
        rows = cent.get_rows(torch.arange(C, device=dev)).double()
        qd = q[:256].double()
        sc = (qd / qd.norm(dim=1, keepdim=True)) @ rows.T / rows.norm(dim=1)[None, :]
        rec.update({"centroid_search_ms": ms_c, "centroid_search_qps": 10_000 / ms_c * 1e3,
                    "centroid_search_ids_identical": bool((torch.topk(sc, 5, dim=1).indices == o3[1][:256]).all().item()),
                    "centroid_search_note": "10^4 x 10^4 x 768: fits L2, no flush between iterations"})
        full.close()
        cent.close()
        return rec

    guarded("C3", c3)

    # ---- C2: 1M x 512 fp32, 10k-query batch, top-10 on one GPU
    def c2():
        if world != 1:
            return None
        n, dim, Q, k = 1_000_000, 512, 10_000, 10
        gal = Gallery(dim, dtype="f32", capacity=n, device=dev.index)
        gen = torch.Generator(dev).manual_seed(2222)
        for s in range(0, n, 250_000):
            gal.upsert(torch.randn(250_000, dim, device=dev, generator=gen))
        gal.set_option("time_k3", 1)
        q = torch.randn(Q, dim, device=dev, generator=gen)
        o2 = (torch.empty((Q, k), dtype=torch.float32, device=dev), torch.empty((Q, k), dtype=torch.int64, device=dev),
              torch.empty((Q, k), dtype=torch.float64, device=dev))
        for _ in range(3):
            gal.search(q, k, out=o2)
        par = parity_check(E, gal, 0, n, q, k, o2)
        ms = E.timed(lambda: gal.search(q, k, out=o2), 10) / 10
        st = gal.search(q, k, out=o2).stats
        tf = 2.0 * Q * n * dim / (st["k3_ms"] / 1e3) / 1e12
        gal.close()
        return {"config": "C2: 1M x 512 fp32, 10k-query batch, top-10, 1 GPU", "value": Q / ms * 1e3, "unit": UNIT,
                "ms_per_step": ms, "k3_ms": st["k3_ms"], "k3_tflops": tf, "k3_frac_of_burst": tf / burst,
                "uncertified_fraction": st["fallback_queries"] / Q, "parity": par,
                "search_operand": "fp16 shadow of the fp32 rows; exact rescoring reads the fp32 master"}

    guarded("C2", c2)

    # ---- distance menu of util/qdrant_manager.py:61-66 beyond COSINE, 1M x 512 fp32, top-10: EUCLID runs on the
    # tensor cores (row-bias epilogue), MANHATTAN on the exact fp64 sweep K5
    def f4():
        if world != 1:
            return None
        n, dim, k = 1_000_000, 512, 10
        rec = {"config": "f4: 1M x 512 fp32, other distances, top-10, 1 GPU"}
        gen = torch.Generator(dev).manual_seed(3333)
        for metric, Q in (("euclid", 10_000), ("manhattan", 256)):
            gal = Gallery(dim, dtype="f32", metric=metric, capacity=n, device=dev.index)
            g2 = torch.Generator(dev).manual_seed(3334)
            for s in range(0, n, 250_000):
                gal.upsert(torch.randn(250_000, dim, device=dev, generator=g2))
            q = torch.randn(Q, dim, device=dev, generator=gen)
            o = (torch.empty((Q, k), dtype=torch.float32, device=dev), torch.empty((Q, k), dtype=torch.int64, device=dev),
                 torch.empty((Q, k), dtype=torch.float64, device=dev))
            gal.search(q, k, out=o)
            ms = E.timed(lambda: gal.search(q, k, out=o), 2) / 2
            rows = gal.get_rows(torch.arange(n, device=dev))
            d = torch.cdist(q[:32].double(), rows.double(), p=2.0 if metric == "euclid" else 1.0)
            same = bool((torch.topk(d, k, dim=1, largest=False).indices == o[1][:32]).all().item())
            r = {"queries": Q, "ms": ms, "qps": Q / ms * 1e3, "ids_identical_to_fp64_cdist": same}
            if metric == "manhattan":
                r["fp64_tflops"] = 2.0 * Q * n * dim / (ms / 1e3) / 1e12
                r["bound"] = ("fp64 CUDA cores (K5): DADD + |.| per (query, row, column); no measured fp64 peak on this "
                              "pool (nominal B200 fp64: ~37 TFLOP/s)")
            else:
                r["tflops"] = 2.0 * Q * n * dim / (ms / 1e3) / 1e12
                r["bound"] = "tensor (K3 with the -|g|^2/2 row bias), of the measured bf16 burst peak"
                r["frac"] = r["tflops"] / burst
            rec[metric] = r
            gal.close()
            del rows, d
        return rec

    guarded("f4", f4)

    # ---- C5: 100M x 768 fp16 over 8 GPUs (12.5M rows = 19.2 GB per GPU), batch sweep 1..65536, top-10
    def c5():
        if not (a.c5 == "on" or (a.c5 == "auto" and world == 8)):
            return None
        g.close()                                         # free the headline gallery (and its fp16 shadow)
        torch.cuda.empty_cache()
        n_total, dim, k = 12_500_000 * world, 768, 10
        t0 = time.perf_counter()
        g5, r05, n5, _ = build_gallery(E, n_total, dim, "f16", 777)
        torch.cuda.synchronize()
        build_s = time.perf_counter() - t0
        offs5 = [shard_range(n_total, r, world)[0] for r in range(world)]
        qgen5 = torch.Generator(dev).manual_seed(555)
        sizes = [1, 2, 4, 8, 16, 32, 64, 128, 256, 512, 1024, 2048, 4096, 8192, 16384, 32768, 65536]
        rows_out = sweep(E, g5, n5, dim, k, sizes, qgen5, offs5, sharded=True, max_iters=20)
        # exactness on a sample: 48 queries against the float64 brute force merged over the shards
        qs = torch.randn(48, dim, device=dev, generator=qgen5)
        S = Searcher(E, g5, 48, k, offs5)
        par = parity_check(E, g5, r05, n5, qs, k, S.device_step(qs), n_check=48)
        # where a single query's latency goes: local search (K3 + finish), then all-gather + K4
        S1 = Searcher(E, g5, 1, k, offs5)
        q1 = torch.randn(1, dim, device=dev, generator=qgen5)
        for _ in range(3):
            S1.device_step(q1)
        loc, k3 = [], []
        for _ in range(20):
            E.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            st = g5.search(q1, k, out=S1.local_out()).stats
            e1.record()
            torch.cuda.synchronize()
            loc.append(e0.elapsed_time(e1))
            k3.append(st["k3_ms"])
        loc_ms, k3_ms_ = E.max_over_ranks(statistics.median(loc)), E.max_over_ranks(statistics.median(k3))
        total1 = rows_out[0]["p50_ms"]
        g5.close()
        return {"config": f"C5: {n_total / 1e6:g}M x 768 fp16 over {world} GPUs ({n5} rows per GPU), top-10, batch sweep",
                "n_gpus": world, "gallery_build_s": round(build_s, 2), "sweep": rows_out, "parity": par,
                "q1_latency_breakdown_ms": {"total_p50": total1, "local_search_p50": loc_ms, "k3_p50": k3_ms_,
                                            "finish_and_host_tail": round(loc_ms - k3_ms_, 4),
                                            "allgather_plus_k4": round(total1 - loc_ms, 4),
                                            "hbm_floor_per_gpu": n5 * dim * 2 / hbm / 1e6}}

    guarded("C5", c5)
    return out


def main():
    a = parse_args()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)


if __name__ == "__main__":
    main()
