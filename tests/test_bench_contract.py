"""bench.py contract checks: the reference arm prints ONE JSON line with the agreed keys, the workload table names
BASELINE.json's configurations, bad arguments are refused, and (on the GPU) --dump-outputs saves the state the timed steps reached."""
import json
import os
import subprocess
import sys

import pytest

from conftest import ROOT


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "cfg1",
                          "--steps", "1", "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["impl"] == "reference" and d["dtype"] == "f64" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["steps"] == 1 and d["warmup"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["value"] > 0


def test_workloads_match_baseline_json():
    sys.path.insert(0, ROOT)
    import bench
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    w4 = bench.WORKLOADS["cfg4"]
    assert (w4["N"], w4["d"], w4["encoding"], w4["kernel"], w4["q"], w4["layers"], w4["outer"], w4["agents"]) == \
        (65536, 4, "yz_cx", "projected", 8, 3, "gaussian", 8)
    assert "N=65536" in base["configs"][3] and "yz_cx" in base["configs"][3]
    w5 = bench.WORKLOADS["cfg5"]
    assert (w5["N"], w5["q"], w5["layers"], w5["agents"], w5["encoding"]) == (131072, 10, 4, 16, "kyriienko")
    w3 = bench.WORKLOADS["cfg3"]
    assert (w3["N"], w3["q"], w3["layers"], w3["agents"], w3["kernel"]) == (16384, 5, 2, 8, "fidelity")
    assert bench.flops_per_entry(w4) == 74 and bench.flops_per_entry(w3) == 259


def test_bad_steps_and_dump_arguments_are_refused(tmp_path):
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path / "out")]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True, timeout=120, cwd=ROOT)
        assert out.returncode == 2 and "error:" in out.stderr, extra
    assert not (tmp_path / "out").exists()


@pytest.mark.gpu
def test_dump_outputs_hold_the_state_after_the_last_timed_step(tmp_path):
    """--dump-outputs writes the ADMM state the timed steps reached (capture() does not advance the run, so warmup + steps
    iterations): equal to the oracle's iterations from the same seeded inputs, and identical from run to run."""
    import numpy as np
    from oracle import agent_step, driver
    sys.path.insert(0, ROOT)
    import bench
    steps, warmup = 2, 1
    runs = []
    for k in range(2):
        out_dir = tmp_path / f"run{k}"
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "cfg1", "--also", "", "--skip-e2e",
                              "--no-cpu-baseline", "--steps", str(steps), "--warmup", str(warmup), "--dump-outputs", str(out_dir)],
                             capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        line = json.loads([l for l in out.stdout.splitlines() if l.strip()][-1])
        assert line["steps"] == steps
        runs.append({name: np.load(out_dir / f"cfg1_{name}.npy") for name in ("z", "theta", "psi", "nll")})
        assert sorted(os.listdir(out_dir)) == sorted(f"cfg1_{name}.npy" for name in runs[-1])
    for name in runs[0]:
        assert runs[0][name].dtype == np.float64 and np.array_equal(runs[0][name], runs[1][name]), name
    w = bench.WORKLOADS["cfg1"]
    x, y = driver.synthetic_dataset(w["N"], w["d"], w["encoding"])
    n_i, A = w["N"] // w["agents"], w["agents"]
    shards = [(x[a * n_i:(a + 1) * n_i], y[a * n_i:(a + 1) * n_i]) for a in range(A)]
    P = runs[0]["z"].size
    rs = np.random.RandomState(42)
    theta, psi = np.round(rs.rand(A, P), 4), np.round(rs.rand(A, P), 4)
    cfg = agent_step.KernelConfig(w["encoding"], w["kernel"], w["q"], w["layers"], w["outer"], training_ignores_outer_kernel=not w["honour_outer"])
    for _ in range(warmup + steps):
        z, theta, psi, res = driver.admm_iteration(cfg, shards, theta, psi, bench.NOISE_STD, bench.RHO, bench.LIP)
    got = runs[0]
    assert got["theta"].shape == (A, P) and got["psi"].shape == (A, P) and got["nll"].shape == (A,)
    assert np.max(np.abs(got["z"] - z)) < 1e-12 and np.max(np.abs(got["theta"] - theta)) < 1e-12
    assert np.max(np.abs(got["psi"] - psi)) < 1e-9
    nll = np.array([r.nll for r in res])
    assert np.max(np.abs(got["nll"] - nll)) < 1e-8 * np.abs(nll).max()
    assert line["final_z_head"] == [float(v) for v in got["z"][:4]]
