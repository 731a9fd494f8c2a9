"""CPU suite for bench.py's contract: the reference arm (the CPU port of the reference's retrieval path, oracle/fast_cpu.py)
runs here without a GPU; its JSON line must carry the keys the driver reads and the SAME `config` object our arm prints
for the same arguments (the driver compares the two arms' configs), and the other ranks of a torchrun launch exit 0
without printing.  Our own arm must refuse to run without a CUDA device instead of falling back to anything."""
import json
import os
import subprocess
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ARGS = ["--rows", "30000", "--dim", "96", "--k", "7", "--steps", "2", "--warmup", "1"]


def _run(extra, env=None):
    e = dict(os.environ, **(env or {}))
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + ARGS + extra, capture_output=True, text=True,
                          timeout=300, env=e, cwd=ROOT)


def _bench_module():
    sys.path.insert(0, ROOT)
    try:
        import bench
    finally:
        sys.path.pop(0)
    return bench


def test_reference_arm_line_and_shared_config():
    r = _run(["--impl", "reference"])
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "queries/s" and d["higher_is_better"] is True
    assert d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 1 and d["vs_baseline"] is None
    assert d["value"] > 0 and abs(d["ms_per_step"] - 1e3 / d["value"]) < 1e-6 * d["ms_per_step"] + 1e-9
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["extrapolated"] is False
    assert cb["rows_timed"] == 30000 and "30000-row corpus" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    bench = _bench_module()
    a = types.SimpleNamespace(rows=30000, dim=96, dtype="bf16", batch=1, k=7)
    assert d["config"] == bench.job_config(a, 1)                  # what our arm prints under "config" for these arguments
    assert d["metric"] == bench.METRIC
    assert set(d["config"]) == {"workload", "rows", "dim", "k", "batch", "parallelism", "l2"}


def test_reference_arm_times_steps_calls_and_dumps_the_last(tmp_path):
    """--steps 2 --warmup 1 times exactly two calls; --dump-outputs writes what the last of them returned."""
    import numpy as np
    from oracle import c_oracle
    r = _run(["--impl", "reference", "--dump-outputs", str(tmp_path)])
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
    assert ", 2 calls, median" in d["cpu_baseline"]["sample"]
    ids, sc = np.load(tmp_path / "batch_1_ids.npy"), np.load(tmp_path / "batch_1_scores.npy")
    assert ids.dtype == np.float64 and sc.dtype == np.float32 and ids.shape == sc.shape == (1, 7)
    bench = _bench_module()
    x = c_oracle.normalize_rows(c_oracle.synth_rows(bench.SEED_CORPUS, 0, 30000, 96), "f32")
    q = c_oracle.synth_rows(bench.SEED_QUERY, 0, 4, 96)[1:2]        # step 1 of 0..1 searches query batch 1
    want_ids, want_sc = c_oracle.cosine_topk(q, x, 7)
    assert np.array_equal(ids, want_ids.astype(np.float64))
    assert np.allclose(sc, want_sc, rtol=1e-5, atol=1e-7)


def test_dump_outputs_samples_queries_within_the_budget(tmp_path):
    import numpy as np
    bench = _bench_module()
    rng = np.random.default_rng(3)
    big_ids = rng.integers(0, 10_000_000, size=(40_000, 200), dtype=np.int64)       # 96 MB as written
    big_sc = rng.random((40_000, 200), dtype=np.float32)
    small_ids, small_sc = big_ids[:4, :10].copy(), big_sc[:4, :10].copy()
    bench.dump_outputs(str(tmp_path), [("batch_4", small_ids, small_sc), ("batch_40000", big_ids, big_sc)])
    assert sum(p.stat().st_size for p in tmp_path.iterdir()) <= 64_000_000
    assert not (tmp_path / "batch_4_queries.npy").exists()
    assert np.array_equal(np.load(tmp_path / "batch_4_ids.npy"), small_ids.astype(np.float64))
    assert np.array_equal(np.load(tmp_path / "batch_4_scores.npy"), small_sc)
    rows = np.load(tmp_path / "batch_40000_queries.npy")
    assert rows.dtype == np.float64 and 0 < len(rows) < 40_000 and (np.diff(rows) > 0).all()
    rows = rows.astype(np.int64)
    assert np.array_equal(np.load(tmp_path / "batch_40000_ids.npy"), big_ids[rows].astype(np.float64))
    assert np.array_equal(np.load(tmp_path / "batch_40000_scores.npy"), big_sc[rows])
    again = tmp_path / "again"
    bench.dump_outputs(str(again), [("batch_4", small_ids, small_sc), ("batch_40000", big_ids, big_sc)])
    assert np.array_equal(np.load(again / "batch_40000_queries.npy"), rows.astype(np.float64))   # the same sample every run


def test_steps_below_one_is_refused():
    r = _run(["--impl", "reference", "--steps", "0"])
    assert r.returncode != 0 and "--steps" in r.stderr


def test_reference_arm_runs_on_rank_0_only():
    r = _run(["--impl", "reference", "--gpus", "2"], env={"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"})
    assert r.returncode == 0 and r.stdout.strip() == ""
    r = _run(["--impl", "reference", "--gpus", "2"], env={"RANK": "0", "LOCAL_RANK": "0", "WORLD_SIZE": "2"})
    assert r.returncode == 0
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["n_gpus"] == 2 and d["config"]["parallelism"] == "row-shard x2"


def test_our_arm_has_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        return                                                     # the GPU suite runs the real thing
    r = _run(["--no-cpu-baseline", "--no-extra-regimes", "--also-batch", "0"])
    assert r.returncode != 0
    assert not [ln for ln in r.stdout.splitlines() if ln.startswith("{")], "a bench line was printed without a GPU"
