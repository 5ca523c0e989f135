"""bench.py's output contract: one JSON line with the keys the driver reads.  The reference arm runs without a GPU
(CPU oracle + the reference's ALGLIB); the B200 arm is checked on the GPU box."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
             "dtype", "data", "config", "e2e", "gpu_launches"}


def _run(args, timeout=600):
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=timeout, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.strip().splitlines() if l.startswith("{")]
    assert len(lines) == 1, res.stdout[-2000:]
    return json.loads(lines[0])


def test_reference_arm_runs_on_the_cpu_alone(have_ref):
    d = _run(["--impl", "reference", "--steps", "1", "--warmup", "0", "--per-gpu", "96"])
    assert BASE_KEYS <= set(d)
    assert d["impl"] == "reference" and d["metric"] == "wbc_control_cycle_solves_per_sec" and d["unit"] == "solves/s"
    assert d["value"] > 0 and d["gpu_launches"] == 0
    assert d["cpu_baseline"]["kind"] == "reference" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"]


@pytest.mark.gpu
def test_b200_arm_json_line():
    d = _run(["--steps", "3", "--warmup", "3", "--no-cpu-baseline"])
    assert BASE_KEYS | {"roofline", "clocks", "p50_ms"} <= set(d)
    assert d["n_gpus"] == 1 and d["steps"] == 3 and d["dtype"] == "f64" and d["scaling"] == "weak"
    assert d["value"] > 1e5 and d["e2e"]["value"] > 1e5 and d["gpu_launches"] == 6
    assert d["e2e"]["h2d_bytes_per_step"] == 4096 * (8 * 93 + 4) and d["e2e"]["d2h_bytes_per_step"] == 4096 * 8 * 18
    r = d["roofline"]
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(r) and 0 < r["frac"] < 1
    assert d["stats"]["solver_failures"] == 0
    assert "sm_mhz" in d["clocks"] and "reasons" in d["clocks"]
    assert "4096" in d["config"]["workload"]


def test_dump_outputs_takes_one_seeded_sample_of_instances_above_the_limit(tmp_path, monkeypatch):
    import bench
    n = 1000
    tau, w = np.arange(12 * n, dtype=np.float64).reshape(12, n), -np.arange(6 * n, dtype=np.float64).reshape(6, n)
    bench.dump_outputs(str(tmp_path / "all"), {"tau": tau, "w": w})
    assert sorted(os.listdir(tmp_path / "all")) == ["tau.npy", "w.npy"]
    assert np.array_equal(np.load(tmp_path / "all" / "tau.npy"), tau)
    monkeypatch.setattr(bench, "DUMP_LIMIT", 40000)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"tau": tau, "w": w})
    keep = np.load(tmp_path / "a" / "instances.npy")
    assert np.array_equal(keep, np.load(tmp_path / "b" / "instances.npy"))
    assert 0 < keep.size < n and sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= 40000
    k = keep.astype(np.int64)
    assert np.array_equal(np.load(tmp_path / "a" / "tau.npy"), tau[:, k]) and np.array_equal(np.load(tmp_path / "a" / "w.npy"), w[:, k])


@pytest.mark.gpu
def test_dump_outputs_are_the_timed_loops_last_step_and_repeat_run_to_run(tmp_path):
    args = ["--warmup", "3", "--no-cpu-baseline", "--no-also"]
    d = _run(args + ["--steps", "2", "--dump-outputs", str(tmp_path / "a")])
    _run(args + ["--steps", "2", "--dump-outputs", str(tmp_path / "b")])
    d3 = _run(args + ["--steps", "3", "--dump-outputs", str(tmp_path / "c")])
    assert d["steps"] == 2 and d3["steps"] == 3
    # the observer state is chained from cycle to cycle: one more timed step moves the estimate, so the dump is the last step's
    assert not np.array_equal(np.load(tmp_path / "a" / "w.npy"), np.load(tmp_path / "c" / "w.npy"))
    assert sorted(os.listdir(tmp_path / "a")) == ["tau.npy", "w.npy"]
    for f, k in (("tau.npy", 12), ("w.npy", 6)):
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype == np.float64 and a.shape == (k, 4096) and np.isfinite(a).all() and np.abs(a).max() > 0
        assert np.array_equal(a, b), f
