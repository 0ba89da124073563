"""CPU: the bench.py contract of the reference arm (`--impl reference`), which runs without a GPU: one JSON line with
the keys the driver reads, the same metric / unit / config as the engine arm, a `cpu_baseline` describing the run and
an `e2e` object repeating the line's value with zero copy bytes (the CPU path moves nothing over PCIe)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference"
    assert d["metric"] == "K*T rollout-steps/s through command()" and d["unit"] == "rollout-steps/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] >= 1
    assert d["dtype"] == "f32" and d["data"] == "synthetic" and d["vs_baseline"] is None and d["scaling"] in ("weak", "strong")
    assert "K=16384 T=30" in d["config"]["workload"]                      # BASELINE.json configs[1]
    assert d["value"] > 0 and abs(d["value"] - 16384 * 30 / (d["ms_per_step"] * 1e-3)) / d["value"] < 1e-6
    cb = d["cpu_baseline"]
    # "reference" when oracle/_ref (the unmodified package, oracle/make_ref.py) is present, else the oracle port
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["unit"] == d["unit"] and cb["value"] == d["value"] and cb["sample"]
    e = d["e2e"]
    assert e["value"] == d["value"] and e["unit"] == d["unit"] and e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0


def test_engine_arm_refuses_to_run_without_a_gpu():
    """No CPU fallback: without a CUDA device the engine arm must fail, not print a number."""
    import torch
    if torch.cuda.is_available():
        return
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--no-cpu-baseline"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode != 0
    assert not any(ln.startswith('{"metric"') for ln in r.stdout.splitlines())


@pytest.mark.gpu
def test_engine_arm_dumps_the_last_timed_command(tmp_path):
    """`--dump-outputs`: what the last timed command() returned to its caller, as .npy files that two runs with the same
    arguments reproduce; `--steps` sets the length of every timed loop."""
    import numpy as np
    outs = []
    for run in range(2):
        d = tmp_path / f"run{run}"
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "nav2d_c3", "--steps", "7",
                            "--warmup", "2", "--no-cpu-baseline", "--dump-outputs", str(d)],
                           capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
        line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
        assert line["steps"] == 7 and line["config"]["step_stats_ms"]["n"] == 7 and line["e2e"]["steps"] == 7
        outs.append({p.stem: np.load(p) for p in d.glob("*.npy")})
    a = outs[0]
    assert sorted(a) == ["U", "action", "cost_total", "theta"]
    assert a["action"].shape == (2,) and a["U"].shape == (40, 2) and a["cost_total"].shape == (8192,) and a["theta"].shape == (5, 2)
    assert all(v.dtype == np.float32 and np.isfinite(v).all() for v in a.values())
    for k in a:
        np.testing.assert_array_equal(a[k], outs[1][k], err_msg=k)


def test_bench_helpers_statistics_bytes_and_workloads():
    """The pure parts of bench.py: trimmed statistics (tests/benchmark_mppi.py:84-113), SURVEY §8(d)'s algorithmic bytes,
    the workload table against BASELINE.json, and the committed traffic file the roofline object reads."""
    sys.path.insert(0, ROOT)
    import bench
    st = bench.trimmed_stats([5.0] + [1.0] * 18 + [0.1])            # one outlier each side: both trimmed away
    assert st["n"] == 20 and st["trimmed_mean"] == 1.0 and st["median"] == 1.0 and st["min"] == 0.1 and st["max"] == 5.0
    assert bench.trimmed_stats([2.0, 4.0])["trimmed_mean"] == 3.0
    c2 = bench.WORKLOADS["pendulum_c2"]
    b_min, b_full = bench.algorithmic_bytes(c2, c2["K"])
    assert (b_min, b_full) == (65784, 2097400)                      # SURVEY §8(d): 4(nx + 2 T nu + K); + 4K + 4 K T nu
    c3 = bench.WORKLOADS["nav2d_c3"]
    assert bench.algorithmic_bytes(c3, c3["K"])[0] == 4 * (2 + 2 * (40 * 2 + 5 * 2) + 8192)    # KMPPI: control points too
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    text = json.dumps(base)
    for name, wl in bench.WORKLOADS.items():
        assert wl["K"] > 0 and wl["T"] > 0 and wl["variant"] in ("mppi", "smppi", "kmppi"), name
    assert "16384" in text and c2["K"] == 16384 and c2["T"] == 30    # the configuration the metric is quoted on
    for name in bench.WORKLOADS:
        t = bench.load_traffic(name)
        assert t is None or (isinstance(t, int) and 10_000 < t < 10_000_000), (name, t)
    assert bench.load_traffic("pendulum_c2") is not None             # the default workload has a committed capture
