"""Cost of batch integrated posterior variance with input gradients (gpp_ipv_points, gpp_nipv_qbatch) on the C4
workload, device-resident.  Arms, alternated after a warm-up, medians of the repeats printed:
  1. ipv_points (U_I and V_I of the integration set, once per factor and set);
  2. nipv_qbatch with the gradient, on the cached set;
  3. posterior_qbatch + posterior_qbatch_grad on the same rows (the floor: the two posterior passes alone).
One call of arm 2 then runs under torch.profiler and the device times of the call and of nipv_block_kernel are
printed.  The card's name and power limit are read in the same run.
Usage: python tools/nipv_probe.py [--repeats R]
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

SIZES = ((512, 4096, 8, 1024), (2048, 1024, 32, 2048), (16384, 128, 128, 4096))  # (N, b, q, M)


def _card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def _kernel_ms(fn, name):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    total = k = 0.0
    for ev in prof.events():
        if ev.device_type != torch.autograd.DeviceType.CUDA:
            continue
        total += ev.device_time / 1e3
        if name in ev.name:
            k += ev.device_time / 1e3
    return total, k


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=5)
    args = ap.parse_args()
    if E.device_count() < 1:
        raise SystemExit("nipv_probe: no CUDA device visible")
    print("card: %s" % _card(), flush=True)
    for n, b, q, M in SIZES:
        X, y = bench.W.c4_workload(n)
        ys = (y - y.min()) / (y.max() - y.min())
        eng = E.Engine(xq=X, y=ys, kernel=E.KERNEL_MATERN52, n_noise=1, n_mean=1, device=0)
        eng.factorize(bench.W.c4_natural(np.zeros(13)))
        dq, m = X.shape[1], b * q
        rs = np.random.RandomState(0)
        xd = torch.from_numpy(rs.rand(m, dq)).cuda()
        xi = torch.from_numpy(rs.rand(M, dq)).cuda()
        vals = torch.empty(b, dtype=torch.float64, device="cuda")
        dx = torch.empty(m, dq, dtype=torch.float64, device="cuda")
        qmean = torch.empty(b, q, dtype=torch.float64, device="cuda")
        qcov = torch.empty(b, q, q, dtype=torch.float64, device="cuda")
        gm0 = torch.zeros(b, q, dtype=torch.float64, device="cuda")
        gc0 = torch.zeros(b, q, q, dtype=torch.float64, device="cuda")

        def points():
            eng.ipv_points(xi)

        def nipv():
            eng.nipv_qbatch(xd, q, out_values=vals, out_d_xq=dx)

        def floor():
            eng.posterior_qbatch(xd, q, out_mean=qmean, out_cov=qcov)
            eng.posterior_qbatch_grad(xd, q, gm0, gc0, out=dx)

        calls = (points, nipv, floor)
        for f in calls:
            f()
        torch.cuda.synchronize()
        ts = {f: [] for f in calls}
        for _ in range(args.repeats):
            for f in calls:
                t0 = time.perf_counter()
                f()
                torch.cuda.synchronize()
                ts[f].append(time.perf_counter() - t0)
        a1, a2, a3 = (statistics.median(ts[f]) * 1e3 for f in calls)
        print("N=%5d b=%5d q=%3d M=%5d: ipv_points %8.2f ms | nipv_qbatch + grad %8.2f ms | "
              "posterior_qbatch + _grad %8.2f ms (nipv %.2fx)" % (n, b, q, M, a1, a2, a3, a2 / a3), flush=True)
        tot, k = _kernel_ms(nipv, "nipv_block_kernel")
        print("    device ms of one nipv_qbatch: total %.2f, nipv_block_kernel %.3f" % (tot, k), flush=True)
        eng.close()
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
