"""Cost of the joint posterior: device-resident gpp_predict against gpp_predict_joint and gpp_sample_posterior on the
same engine (C4 workload, candidates and outputs on the GPU).

For each (N, m) the three calls alternate after a warm-up, and the medians of the repeats are printed with their
ratios to predict.  One sample_posterior call per size then runs under torch.profiler; its kernels are split into
stages at the launches that open them (U = J1 up to the last predict_finish_kernel, K** from joint_diag_kernel, SYRK =
the GEMM after the last K** tile, potrf_blocked from the first leaf, draws from fill_rows_kernel; the jitter ladder
adds its retries to K**, SYRK and potrf).  The split relies on those kernel names (joint_diag_kernel,
dgemm_dmma_kernel, leaf_potrf_trinv_kernel, fill_rows_kernel): renaming one of them moves its time into the previous
stage.  The stages are converted to FP64 rates from the shapes (U m N^2, SYRK m^2 N, factor m^3 / 3, draws S m^2
flop) and compared with the DMMA GEMM probe (gpp_probe_dgemm) of the same run.  The card's name and power limit are read in the same run.
Usage: python tools/joint_posterior_probe.py [--repeats R] [--samples S]
"""
import argparse
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "gp-plus_b200")]

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from gpplus_b200 import _engine as E  # noqa: E402

SIZES = ((512, 4096), (2048, 8192), (16384, 4096), (16384, 16384))
STAGES = ("U", "K**", "SYRK", "potrf", "draws")


def _card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def _stage_times(fn):
    """device milliseconds of each stage of one call, from the kernel trace"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    evs = sorted((ev for ev in prof.events() if ev.device_type == torch.autograd.DeviceType.CUDA
                  and "memcpy" not in ev.name.lower() and "memset" not in ev.name.lower()),
                 key=lambda ev: ev.time_range.start)
    tot = dict.fromkeys(STAGES, 0.0)
    stage = "U"
    for ev in evs:
        name = ev.name
        if "joint_diag_kernel" in name:
            stage = "K**"
        elif "dgemm_dmma" in name and stage == "K**":
            stage = "SYRK"
        elif "leaf_potrf" in name and stage in ("K**", "SYRK"):
            stage = "potrf"
        elif "fill_rows_kernel" in name:
            stage = "draws"
        tot[stage] += ev.device_time / 1e3
    return tot


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--samples", type=int, default=1024)
    args = ap.parse_args()
    if E.device_count() < 1:
        raise SystemExit("joint_posterior_probe: no CUDA device visible")
    print("card: %s" % _card(), flush=True)
    g = 8192
    ms = E.probe_dgemm(g, g, g, iters=5)
    dgemm = 2.0 * g ** 3 / (ms * 1e-3) / 1e12
    print("gpp_probe_dgemm %d^3: %.2f ms, %.1f TFLOP/s" % (g, ms, dgemm), flush=True)
    S = args.samples
    for n, m in SIZES:
        X, y = bench.W.c4_workload(n)
        ys = (y - y.min()) / (y.max() - y.min())
        eng = E.Engine(xq=X, y=ys, kernel=E.KERNEL_MATERN52, n_noise=1, n_mean=1, device=0)
        eng.factorize(bench.W.c4_natural(np.zeros(13)))
        dq = X.shape[1]
        xd = torch.from_numpy(np.random.RandomState(0).rand(m, dq)).cuda()
        base = torch.from_numpy(np.random.RandomState(1).standard_normal((S, m))).cuda()
        mu, var = (torch.empty(m, dtype=torch.float64, device="cuda") for _ in range(2))
        cov = torch.empty(m, m, dtype=torch.float64, device="cuda")
        draws = torch.empty(S, m, dtype=torch.float64, device="cuda")
        jit = []

        def plain():
            eng.predict(xd, out_mean=mu, out_var=var)

        def joint():
            eng.predict_joint(xd, out_mean=mu, out_cov=cov)

        def sample():
            jit.append(eng.sample_posterior(xd, base, out=draws)[1])

        for f in (plain, joint, sample):
            f()
        torch.cuda.synchronize()
        ts = {plain: [], joint: [], sample: []}
        for _ in range(args.repeats):
            for f in (plain, joint, sample):
                t0 = time.perf_counter()
                f()
                torch.cuda.synchronize()
                ts[f].append(time.perf_counter() - t0)
        p, j, s = (statistics.median(ts[f]) * 1e3 for f in (plain, joint, sample))
        st = _stage_times(sample)
        flop = {"U": float(m) * n * n, "SYRK": float(m) * m * n, "potrf": float(m) ** 3 / 3, "draws": float(S) * m * m}
        print("N=%5d m=%5d S=%d dq=%d jitter=%g: predict %8.2f ms  predict_joint %8.2f ms (%.2fx)  "
              "sample_posterior %8.2f ms (%.2fx)" % (n, m, S, dq, max(jit), p, j, j / p, s, s / p), flush=True)
        print("    stages of sample_posterior (device ms): " + "  ".join(
            "%s %.2f" % (k, st[k]) + (" [%.1f TFLOP/s, %.2f of DGEMM]" % (flop[k] / st[k] / 1e9, flop[k] / st[k] / 1e9
                                                                         / dgemm)
                                       if k in flop and st[k] > 0 else "") for k in STAGES), flush=True)
        eng.close()
        del cov, draws, base
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
