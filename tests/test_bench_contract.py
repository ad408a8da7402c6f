"""CPU: the reference arm of bench.py (the oracle port timed on the host cores) prints exactly ONE JSON line on stdout
with the keys of the contract -- the GPU arm shares `emit()` and `workload_config()` with it."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    env = dict(os.environ, OMP_NUM_THREADS="1")          # what torchrun exports; the arm must still use every core
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, env=env, timeout=300)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "solves/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["vs_baseline"] is None and d["dtype"] == "f64"
    assert "workload" in d["config"] and "n=10" in d["config"]["workload"] and "N=6" in d["config"]["workload"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["value"] == d["value"] and cb["cores"] >= 1 and "sample" in cb
    assert cb["cores"] == len(os.sched_getaffinity(0))
    assert d["e2e"] == {"value": d["value"], "unit": "solves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                        "--warmup", "0"], capture_output=True, text=True, env=env, timeout=120)
    assert p.returncode == 0 and p.stdout.strip() == ""


def test_dump_outputs_writes_float64_and_one_shared_sample_above_the_limit(tmp_path):
    """bench.dump_outputs (--dump-outputs): every array whole while they fit, else the same seeded problems of each
    array (indices in sample_index.npy), within the byte limit and identical from call to call."""
    import importlib
    import numpy as np
    import torch
    bench = importlib.import_module("bench")
    B = 1000
    arrays = {"obj": torch.arange(B, dtype=torch.float64), "u": torch.arange(B * 6, dtype=torch.float64).reshape(B, 6),
              "status": torch.full((B,), 2, dtype=torch.int32)}
    bench.dump_outputs(str(tmp_path / "all"), arrays)
    assert sorted(p.name for p in (tmp_path / "all").iterdir()) == ["obj.npy", "status.npy", "u.npy"]
    for name, a in arrays.items():
        d = np.load(tmp_path / "all" / f"{name}.npy")
        assert d.dtype == np.float64 and np.array_equal(d, a.numpy())
    limit = 40_000
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), arrays, limit_bytes=limit)
    files = sorted((tmp_path / "a").iterdir())
    assert sum(p.stat().st_size for p in files) <= limit
    idx = np.load(tmp_path / "a" / "sample_index.npy").astype(np.int64)
    assert 0 < len(idx) < B and (np.diff(idx) > 0).all()
    assert np.array_equal(np.load(tmp_path / "a" / "obj.npy"), idx) and (np.load(tmp_path / "a" / "status.npy") == 2).all()
    assert np.array_equal(np.load(tmp_path / "a" / "u.npy"), arrays["u"].numpy()[idx])
    for p in files:
        assert np.array_equal(np.load(p), np.load(tmp_path / "b" / p.name))


def test_episode_legs_warm_up_at_full_size_and_report_the_median():
    """bench._episodes: one untimed run first (idle clocks, cold allocator), then the median of the timed runs, each
    bracketed by the caller's sync and reduced over the ranks by the caller's reduction."""
    import importlib
    import time as _time
    bench = importlib.import_module("bench")
    calls, syncs = [], []
    durations = iter([0.0, 0.03, 0.01, 0.02])               # warm-up, then three timed runs

    def run():
        calls.append(len(calls))
        _time.sleep(next(durations))
        return len(calls)

    out, med, runs = bench._episodes(run, reps=3, sync=lambda: syncs.append(1), reduce=lambda d: round(d, 2))
    assert calls == [0, 1, 2, 3] and out == 4               # warm-up + 3 timed; the last result is returned
    assert len(syncs) == 3 and len(runs) == 3
    assert med == sorted(runs)[1] and min(runs) <= med <= max(runs)
