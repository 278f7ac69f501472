"""bench.py's output contract, checked on the arm that runs without a GPU (the CPU reference arm), and the
``--dump-outputs`` files of both arms."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _last_step_oracle(n, steps):
    """Oracle result at the theta of the last of ``steps`` timed steps of rank 0."""
    sys.path.insert(0, ROOT)
    import bench
    import bench_workloads as W
    from oracle import gp_oracle as O
    thetas = W.c4_theta_points(W.c4_model(256))
    return O.mll(W.c4_oracle_problem(n), W.c4_natural(bench.step_theta(thetas, steps - 1)), want_grad=True)


def _load_dump(path):
    got = {f[:-4]: np.load(os.path.join(path, f)) for f in os.listdir(path) if f.endswith(".npy")}
    assert got and all(v.dtype == np.float64 for v in got.values())
    return got


def test_reference_arm_prints_one_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--n", "256", "--steps",
                          "1", "--warmup", "0"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "evals/s" and d["higher_is_better"] is True
    assert d["metric"] == "MLL+grad evals/sec (N=16k, fp64)" and d["dtype"] == "f64" and d["vs_baseline"] is None
    assert d["value"] > 0 and d["config"]["workload"].startswith("synthetic exact GP N=256")
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # the steps reported are the evaluations really run at the FULL size (no extrapolation), and they fit the run
    assert d["steps"] == 1 and d["steps_requested"] == 1 and d["warmup"] == 0
    assert abs(d["ms_per_step"] * d["steps"] * 1e-3 - d["steps"] / d["value"]) < 1e-6
    # both arms print the same config object
    sys.path.insert(0, ROOT)
    import bench
    assert d["config"] == bench.bench_config(256)


def test_reference_arm_dumps_its_last_step(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--n", "256", "--steps",
                          "2", "--warmup", "0", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][0])
    assert d["steps"] == 2
    got, ref = _load_dump(tmp_path), _last_step_oracle(256, 2)
    assert set(got) == set(ref)
    for k, v in ref.items():
        np.testing.assert_allclose(got[k], v, rtol=1e-10, atol=0, err_msg=k)


@pytest.mark.gpu
def test_our_arm_dumps_its_last_timed_step(tmp_path):
    n, steps = 4096, 3
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--n", str(n), "--steps", str(steps),
                          "--warmup", "3", "--no-extras", "--no-cpu-baseline", "--no-dmma-arm", "--no-prior-sweep",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][0])
    assert d["steps"] == steps
    got, ref = _load_dump(tmp_path), _last_step_oracle(n, steps)
    assert set(got) == set(ref) | {"objective_value", "objective_grad"}
    assert abs(float(got["nll"]) - ref["nll"]) <= 1e-9 * abs(ref["nll"])
    assert float(got["jitter"]) == ref["jitter"]
    g = np.concatenate([got["d_w"], [got["d_sigma_f2"]], got["d_noise"], got["d_beta"]])
    gr = np.concatenate([ref["d_w"], [ref["d_sigma_f2"]], ref["d_noise"], ref["d_beta"]])
    assert np.max(np.abs(g - gr)) <= 1e-8 * np.max(np.abs(gr))
    # (value, gradient) of the public objective at the same theta: the model-level oracle of MLLObjective.fun
    import bench
    import bench_workloads as W
    from oracle import gpplus_oracle as GO
    X, y = W.c4_workload(n)
    theta = bench.step_theta(W.c4_theta_points(W.c4_model(256)), steps - 1)
    f_ref, g_ref = GO.neg_log_posterior({"X": X, "y": y, "kernel": "Matern52Kernel"}, theta)
    assert got["objective_value"].shape == () and got["objective_grad"].shape == g_ref.shape
    assert abs(float(got["objective_value"]) - f_ref) <= 1e-9 * abs(f_ref)
    assert np.max(np.abs(got["objective_grad"] - g_ref)) <= 1e-7 * np.max(np.abs(g_ref))


def test_reference_arm_is_silent_on_other_ranks():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--n",
                          "256"], capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_our_arm_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        return
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1"], capture_output=True, text=True,
                         timeout=300, cwd=ROOT)
    assert out.returncode != 0 and "no CUDA device" in (out.stderr + out.stdout)
