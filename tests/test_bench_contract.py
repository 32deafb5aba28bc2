"""bench.py's reference arm is CPU-only, so its JSON line -- the same contract the B200 arm prints -- can be checked
here: one line on stdout, the keys the driver reads, the CPU baseline described, no GPU work claimed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DUMPED = ("scores", "rows", "scores64")


def test_reference_arm_prints_one_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches", "impl"):
        assert key in d, key
    assert d["impl"] == "reference" and d["steps"] == 1 and d["warmup"] == 0 and d["n_gpus"] == 1
    assert d["metric"] == "top-10 cosine queries/s on 10M x 768" and d["unit"] == "queries/s"
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0 and d["value"] > 0
    lit = d["reference_literal"]                              # B1 / B3: the reference's own per-pair and per-class loops
    assert lit["B1_cosine_similarity_pairs_per_s"] > 0 and lit["B3_compute_average_classes_per_s"] > 0


def test_non_zero_ranks_of_the_reference_arm_exit_without_work():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1", MASTER_ADDR="127.0.0.1", MASTER_PORT="29999")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_dump_outputs_writes_float_arrays_and_samples_past_the_limit(tmp_path):
    import bench

    rng = np.random.default_rng(3)
    Q, k = 500, 7
    s64 = -np.sort(-rng.random((Q, k)), axis=1)
    rows = rng.integers(0, 10**12, (Q, k))
    bench.dump_outputs(str(tmp_path / "all"), s64.astype(np.float32), rows, s64)
    got = {n: np.load(tmp_path / "all" / f"{n}.npy") for n in DUMPED}
    assert [got[n].dtype for n in DUMPED] == [np.float32, np.float64, np.float64]
    assert np.array_equal(got["rows"].astype(np.int64), rows) and np.array_equal(got["scores64"], s64)
    assert not (tmp_path / "all" / "query_index.npy").exists()
    limit = 4096 + 100 * (k * (4 + 8 + 8) + 8)                   # room for 100 queries
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), s64.astype(np.float32), rows, s64, limit=limit)
    idx = np.load(tmp_path / "a" / "query_index.npy")
    assert idx.shape == (100,) and np.all(np.diff(idx) > 0)
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= limit
    for n in DUMPED + ("query_index",):
        assert np.array_equal(np.load(tmp_path / "a" / f"{n}.npy"), np.load(tmp_path / "b" / f"{n}.npy"))
    assert np.array_equal(np.load(tmp_path / "a" / "rows.npy"), rows[idx.astype(np.int64)].astype(np.float64))


def test_no_timed_steps_and_dumps_without_the_headline_search_are_refused():
    for args in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"], ["--sweep", "8", "--dump-outputs", "out"]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                             timeout=300, cwd=ROOT)
        assert out.returncode == 2 and out.stdout == "", (args, out.stderr)


@pytest.mark.gpu
def test_two_runs_with_the_same_arguments_dump_the_same_outputs(tmp_path):
    args = ["--rows", "30000", "--queries", "200", "--k", "10", "--steps", "2", "--warmup", "1", "--no-configs",
            "--no-cpu-baseline"]
    dumps = []
    for run in ("a", "b"):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args, "--dump-outputs", str(tmp_path / run)],
                             capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        line = json.loads(out.stdout)
        assert line["steps"] == 2 and line["parity"]["ids_identical"]
        dumps.append({n: np.load(tmp_path / run / f"{n}.npy") for n in DUMPED})
    for n in DUMPED:
        assert dumps[0][n].shape == (200, 10) and np.array_equal(dumps[0][n], dumps[1][n]), n
    rows, s64 = dumps[0]["rows"], dumps[0]["scores64"]
    assert np.all((rows >= 0) & (rows < 30000)) and np.all(np.diff(s64, axis=1) <= 0)
    assert np.allclose(dumps[0]["scores"], s64, rtol=0, atol=1e-6)
