"""bench.py contract (CPU part): the reference arm prints ONE JSON line with the keys the driver reads."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_line_has_the_contract_keys():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--rows", "20000", "--dim", "64",
                          "--cpu-sample", "20000", "--cpu-queries", "300", "--steps", "2", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "impl", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["impl"] == "reference" and d["steps"] == 2 and d["warmup"] == 1 and d["higher_is_better"] is True
    assert d["metric"] == "ann_search_qps_at_recall10_ge_0.95" and d["unit"] == "queries/s" and d["value"] > 0
    assert d["vs_baseline"] is None and d["data"] == "synthetic" and "workload" in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["recall_at_10"] >= 0.95
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_our_arm_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        return
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--rows", "1000", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode != 0                      # no CPU fallback on the product path
    assert not any(ln.startswith("{") for ln in out.stdout.splitlines())


def test_committed_bench_lines_carry_the_contract_keys():
    """The bench lines committed under profiles/ (what BASELINE.md quotes) have every key the measurement contract names,
    and their roofline arithmetic is self-consistent: achieved = algorithmic bytes per launch / kernel time."""
    import json
    for name in ("r2_bench_c3_n1.json", "r2_bench_c3_n8.json", "r2_bench_c2_n1.json"):
        d = json.load(open(os.path.join(ROOT, "profiles", name)))
        for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                    "vs_baseline", "dtype", "data", "config", "clocks", "e2e", "gpu_launches", "roofline"):
            assert key in d, (name, key)
        assert d["metric"] == "ann_search_qps_at_recall10_ge_0.95" and d["higher_is_better"] is True
        assert "workload" in d["config"] and "model" not in d["config"]
        assert d["config"]["recall_at_10"] >= 0.95
        assert d["gpu_launches"] > 0 and d["vs_baseline"] is None
        e = d["e2e"]
        assert e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0 and 0 < e["value"] <= d["value"] * 1.02
        r = d["roofline"]
        assert r["bound"] == "hbm" and r["unit"] == "GB/s"
        achieved = r["algorithmic_bytes_per_launch"] / (r["kernel_ms_per_launch"] * 1e-3) / 1e9
        assert abs(achieved - r["achieved"]) / r["achieved"] < 1e-6
        assert abs(r["achieved"] / r["peak"] - r["frac"]) < 1e-9 and 0.3 < r["frac"] < 1.1
        # the kernel cannot take longer than the step it is part of
        batches = int(d["config"]["step"].split()[0])
        assert r["kernel_ms_per_launch"] * batches <= d["ms_per_step"] * 1.001
        if d["n_gpus"] == 1:
            cb = d["cpu_baseline"]
            assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] > 0 and "sample" in cb
            assert d["build_roofline"]["tensor"]["frac"] > 0 and d["build_roofline"]["hbm"]["frac"] > 0


def _dumped(d):
    import numpy as np
    out = {name: np.load(os.path.join(d, name + ".npy")) for name in ("keys", "distances", "query_rows")}
    assert out["keys"].dtype == np.float64 and out["distances"].dtype == np.float32 and out["query_rows"].dtype == np.float64
    assert out["keys"].shape == out["distances"].shape and out["query_rows"].shape == out["keys"].shape[:1]
    assert sum(os.path.getsize(os.path.join(d, f)) for f in os.listdir(d)) <= 64 << 20
    return out


def test_reference_arm_dumps_what_its_last_step_returned(tmp_path):
    """--dump-outputs: the keys and distances of the last timed search, for every query of the step."""
    import numpy as np
    import oracle as O
    from importlib import import_module
    ds = import_module("vector_store_b200.host.datasets")
    d = str(tmp_path / "out")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--rows", "20000", "--dim", "64",
                          "--cpu-sample", "20000", "--cpu-queries", "300", "--steps", "2", "--warmup", "1", "--dump-outputs", d],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    got = _dumped(d)
    assert got["keys"].shape == (300, 10) and np.array_equal(got["query_rows"], np.arange(300))
    assert np.all(np.diff(got["distances"], axis=1) >= 0)
    # the bench's corpus and queries (16 mixture components at 20 000 rows); the arm tuned its ef to recall@10 >= 0.95
    x = ds.embedding_mix(20000, 64, seed=1234, n_clusters=16)
    q = ds.embedding_mix(300, 64, seed=4321, n_clusters=16)
    tk, _, _, _ = O.exact_topk(x, q, 10, O.COS, O.F32, keys=np.arange(20000, dtype=np.uint64))
    assert O.recall_at_k(got["keys"].astype(np.uint64), tk) >= 0.9


def test_dump_outputs_samples_above_the_budget(tmp_path):
    import numpy as np
    import bench
    keys = np.arange(1000 * 10, dtype=np.uint64).reshape(1000, 10)
    keys[3, 9] = np.uint64(0xFFFFFFFFFFFFFFFF)
    dists = np.sort(np.random.default_rng(1).random((1000, 10)).astype(np.float32), axis=1)
    bench.dump_outputs(str(tmp_path / "all"), keys, dists)
    got = _dumped(str(tmp_path / "all"))
    assert np.array_equal(got["keys"][:3], keys[:3].astype(np.float64)) and got["keys"][3, 9] == 2.0 ** 64
    assert np.array_equal(got["distances"], dists) and np.array_equal(got["query_rows"], np.arange(1000))
    budget = 1024 + 300 * (10 * 12 + 8)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), keys, dists, budget=budget)
    a, b = _dumped(str(tmp_path / "a")), _dumped(str(tmp_path / "b"))
    assert a["keys"].shape == (300, 10) and sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= budget
    rows = a["query_rows"].astype(np.int64)
    assert np.all(np.diff(rows) > 0) and np.array_equal(a["keys"], keys[rows].astype(np.float64))
    assert np.array_equal(a["distances"], dists[rows])
    assert all(np.array_equal(a[n], b[n]) for n in a)                  # a fixed sample: the same rows every run


@pytest.mark.gpu
def test_our_arm_dumps_every_batch_of_its_last_step(tmp_path):
    """--dump-outputs on the timed device path: one row per query of the last step's batches (batch j searches the
    query pool's batch j % 4), the hits are the oracle's nearest neighbours of those queries, and a second run with the
    same arguments (the graph build streams the rows beyond its 131 072-row all-pairs prefix) writes the same arrays."""
    import numpy as np
    import oracle as O
    from importlib import import_module
    ds = import_module("vector_store_b200.host.datasets")
    n, dim, B, R, k = 200_000, 128, 2000, 3, 10
    runs = []
    for run in ("a", "b"):
        d = str(tmp_path / run)
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--rows", str(n), "--dim", str(dim), "--batch",
                              str(B), "--batches-per-step", str(R), "--steps", "2", "--warmup", "1", "--search-width", "2",
                              "--no-cpu-baseline", "--dump-outputs", d], capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        line = json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("{")][-1])
        assert line["steps"] == 2
        runs.append(_dumped(d))
    got = runs[0]
    assert all(np.array_equal(got[name].view(np.uint64 if got[name].dtype == np.float64 else np.uint32),
                              runs[1][name].view(np.uint64 if got[name].dtype == np.float64 else np.uint32)) for name in got)
    assert got["keys"].shape == (R * B, k) and np.array_equal(got["query_rows"], np.arange(R * B))
    assert np.all(np.diff(got["distances"], axis=1) >= 0) and np.all(got["keys"] < n)
    clusters = 51                                                         # 256 per million rows
    x = ds.embedding_mix(n, dim, seed=1234, n_clusters=clusters)
    sel = np.arange(0, B, 40)
    for j in range(R):
        q = ds.embedding_mix(B, dim, seed=4321 + j, n_clusters=clusters)[sel]
        tk, td, _, _ = O.exact_topk(x, q, k, O.COS, O.BF16, keys=np.arange(n, dtype=np.uint64))
        assert O.recall_at_k(got["keys"][j * B + sel].astype(np.uint64), tk) >= 0.9, j
        first = got["keys"][j * B + sel, 0] == tk[:, 0]                   # a shared top-1 carries the oracle's distance
        assert first.mean() >= 0.9 and np.array_equal(got["distances"][j * B + sel, 0][first], td[first, 0])


def test_steps_below_one_are_refused():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode != 0 and "--steps" in out.stderr


def test_reference_arm_under_torchrun_prints_one_line_from_rank_0():
    """The driver launches the reference arm like our arm (torchrun for N > 1): rank 0 alone runs and prints, the other
    ranks exit 0 without work."""
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29533", os.path.join(ROOT, "bench.py"),
                          "--impl", "reference", "--gpus", "2", "--rows", "20000", "--dim", "64", "--cpu-sample", "20000",
                          "--cpu-queries", "200", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["cpu_baseline"]["kind"] == "port" and d["e2e"]["h2d_bytes_per_step"] == 0
