"""bench.py prints ONE JSON line with the keys the driver reads (CPU: reference arm; GPU: b200 arm)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config"}


def _run(args, timeout=600):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True,
                       timeout=timeout, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, r.stdout
    return json.loads(lines[0])


def test_reference_arm_line():
    d = _run(["--impl", "reference", "--workload", "mnist_cnn", "--steps", "8", "--warmup", "3", "--cpu-budget", "1"])
    assert BASE_KEYS <= set(d) and d["impl"] == "reference" and d["higher_is_better"] is True
    assert d["unit"] == "micro-steps/s" and d["value"] > 0 and d["vs_baseline"] is None and d["dtype"] == "f32"
    assert "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_nonzero_rank_prints_nothing():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                       capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


@pytest.mark.gpu
def test_b200_arm_line():
    d = _run(["--workload", "mnist_cnn", "--steps", "40", "--warmup", "3", "--e2e-steps", "8", "--cpu-budget", "1"])
    assert BASE_KEYS <= set(d) and d["impl"] == "b200" and d["n_gpus"] == 1 and d["steps"] == 40 and d["warmup"] >= 3
    assert d["scaling"] == "weak" and d["data"] == "synthetic" and d["dtype"] == "f32" and d["gpu_launches"] == 40
    rf = d["roofline"]
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(rf) and rf["bound"] == "hbm" and rf["unit"] == "GB/s"
    assert abs(rf["frac"] - rf["achieved"] / rf["peak"]) < 1e-9
    e = d["e2e"]
    assert e["value"] > 0 and e["h2d_bytes_per_step"] == 4 * d["config"]["P"] and e["d2h_bytes_per_step"] > 0
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"])
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] > 0
    assert "l2" in d["config"] and "workload" in d["config"]
    # exact window mix: 40 steps at N=4 are 10 applies + 30 accumulates, and the line says so
    assert d["config"]["apply_launches"] == 10 and d["config"]["accumulate_launches"] == 30 and d["config"]["window_exact"] is True
    # the pre-timing parity self-check ran against the oracle and passed
    assert d["parity"]["ok"] is True and d["parity"]["max_rel_err"] <= 1e-5 and d["parity"]["world"] == 1


@pytest.mark.gpu
def test_b200_arm_dumps_the_last_timed_step(tmp_path):
    """--dump-outputs: float32 arrays within 64 MB, identical for identical arguments, and they follow --steps."""
    import numpy as np
    base = ["--workload", "mnist_cnn", "--warmup", "3", "--e2e-steps", "0", "--model-steps", "0", "--cpu-budget", "0",
            "--parity-steps", "0"]
    runs = {}
    for tag, steps in (("a", 8), ("b", 8), ("c", 12)):
        d = _run(base + ["--steps", str(steps), "--dump-outputs", str(tmp_path / tag)])
        assert d["steps"] == steps and d["config"]["apply_launches"] == steps // 4
        runs[tag] = {n: np.load(tmp_path / tag / f"{n}.npy") for n in ("param", "adam_m", "adam_v", "accum", "stats")}
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= 64 << 20
    a, b, c = runs["a"], runs["b"], runs["c"]
    P = d["config"]["P"]
    for n in ("param", "adam_m", "adam_v", "accum"):
        assert a[n].dtype == np.float32 and a[n].shape == (P,)
    assert a["stats"].dtype == np.float32 and a["stats"][0] == 1.0      # 8 steps at N=4 end on an apply
    assert not a["accum"].any()                                            # ... which zeroes the accumulators
    for n in a:
        assert np.array_equal(a[n], b[n]), n
    assert not np.array_equal(a["param"], c["param"])                     # one more window moved the parameters


def test_dump_outputs_and_steps_are_validated():
    for args in (["--impl", "reference", "--dump-outputs", "out"], ["--steps", "0"]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True,
                           timeout=120, cwd=ROOT)
        assert r.returncode == 2 and "error" in r.stderr and r.stdout == ""


def test_both_arms_print_the_same_metric_string():
    """The driver divides the two arms only when `metric` matches: one constant feeds both lines."""
    import re
    src = open(os.path.join(ROOT, "bench.py")).read()
    assert len(re.findall(r'"metric": METRIC', src)) >= 2 and '"impl": "b200"' in src and '"impl": "reference"' in src


@pytest.mark.parametrize("N", [1, 2, 3, 4, 5, 6, 8, 32])
def test_rotation_phases_give_one_apply_per_window(N):
    """bench.py steps R rotating state sets round-robin; the per-set global_step phases must put exactly one
    apply (pre-increment step % N == 0, optimization.py:91) at bench steps i % N == N-1 and nowhere else."""
    sys.path.insert(0, ROOT)
    import bench
    R = bench.rotation_for(N)
    assert R >= 3
    gs = [bench.set_start_step(r, R, N) for r in range(R)]
    for i in range(6 * N * R):
        r = i % R
        applies = (gs[r] % N) == 0
        gs[r] += 1
        assert applies == (i % N == N - 1), (N, R, i)
