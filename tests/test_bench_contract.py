"""bench.py's output contract: exactly one JSON line on stdout with the keys the driver reads."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e", "cpu_baseline"}


def _run(*flags, timeout=600):
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *flags], capture_output=True, text=True,
                         timeout=timeout, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    return json.loads(lines[0])


def test_reference_arm_line():
    d = _run("--impl", "reference", "--steps", "1", "--warmup", "1", "--cpu-step-seconds", "0.5")
    assert d["impl"] == "reference" and BASE_KEYS <= set(d)
    assert d["metric"] == "hyp x point evals/sec (fp64)" and d["unit"] == "evals/s" and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] == d["value"] > 0
    assert d["e2e"] == {"value": d["value"], "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["vs_baseline"] is None and d["dtype"] == "f64"


@pytest.mark.gpu
def test_native_arm_line():
    d = _run("--steps", "2", "--warmup", "3", "--cpu-baseline-seconds", "1")
    assert BASE_KEYS | {"roofline", "clocks", "gpu_launches"} <= set(d)
    assert d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 3 and d["scaling"] == "weak" and d["data"] == "synthetic"
    assert d["value"] > 5e11 and d["e2e"]["value"] > 5e11 and d["e2e"]["h2d_bytes_per_step"] >= 3_200_000
    r = d["roofline"]
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(r) and 0.5 < r["frac"] < 1.2
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and r["unit"] == "TFLOP/s"
    assert d["gpu_launches"] >= 2 * 6 and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["kind"] == "port"
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"])
    assert "workload" in d["config"] and "config3" in d["config"]["workload"]


def test_argument_errors():
    for flags in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *flags], capture_output=True, text=True,
                             timeout=120, cwd=ROOT)
        assert out.returncode == 2 and not out.stdout and "error" in out.stderr, flags


@pytest.mark.gpu
def test_dump_outputs_is_the_last_timed_step(engine, tmp_path):
    """--dump-outputs writes the results of the last timed step: config 2's scene with the device sampler seeded by
    the step index, so with --steps 3 the estimate of seed 2."""
    import numpy as np

    from structure_from_motion_b200.scenes import make_scene

    d = _run("--workload", "config2", "--steps", "3", "--warmup", "1", "--no-cpu-baseline", "--no-e2e",
             "--no-fp32-variant", "--dump-outputs", str(tmp_path / "out"))
    assert d["steps"] == 3
    got = {p.stem: np.load(p) for p in (tmp_path / "out").glob("*.npy")}
    assert all(a.dtype == np.float64 and np.isfinite(a).all() for a in got.values())
    assert sum(p.stat().st_size for p in (tmp_path / "out").iterdir()) <= 64 * 10 ** 6
    K, x1, x2, *_ = make_scene(10_000, 0.4, seed=0)
    engine.upload_pairs(x1, x2, K)
    engine.sample_device(2, 16_384)
    best, _, _, poses, num, idx, ok, X = engine.two_view(1.5e-6, 10, "rms", "min_error", 50.0, want_mask=False,
                                                         want_sed=False)
    assert got["best_index"] == best.index and got["best_err"] == best.err and got["count_extra"] == best.count_extra
    assert np.array_equal(got["E"].reshape(9), np.array(best.E)) and got["num_inliers"] == num
    assert np.array_equal(got["inlier_idx"], idx) and np.array_equal(got["pass_bits"], ok)
    passing = ((ok >> poses.best) & 1).astype(bool)  # the library's rows for the other inliers are NaN
    assert passing.any() and np.isnan(X[~passing]).all() and np.array_equal(got["points"], X[passing])
    assert got["pose_best"] == poses.best and got["pose_counts"].tolist() == list(poses.counts)
    assert np.array_equal(got["pose_R"].reshape(4, 9), np.array(poses.R))
