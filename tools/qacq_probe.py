"""Cost of Monte-Carlo batch acquisition with input gradients (gpp_acq_qbatch) on the C4 workload, device-resident,
against two other ways of getting the same numbers on the same engine:
  1. acquisition_qbatch with the gradient (one call);
  2. posterior_qbatch + posterior_qbatch_grad (the floor: the two posterior passes alone, no sampling);
  3. the host path: posterior_qbatch to the host, the MC step in torch with autograd through the batched Cholesky,
     then posterior_qbatch_grad with the upstream gradients.
The three arms alternate after a warm-up and the medians of the repeats are printed.  One call of arm 1 then runs
under torch.profiler and the device time of qacq_mc_kernel is printed.  The card's name and power limit are read in
the same run.
Usage: python tools/qacq_probe.py [--repeats R]
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
from gpplus_b200.models.gpregression import sobol_normal_samples  # noqa: E402

SIZES = ((512, 4096, 8, 512), (2048, 1024, 32, 512), (16384, 128, 128, 512))


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
        raise SystemExit("qacq_probe: no CUDA device visible")
    print("card: %s" % _card(), flush=True)
    for n, b, q, S in SIZES:
        X, y = bench.W.c4_workload(n)
        ys = (y - y.min()) / (y.max() - y.min())
        eng = E.Engine(xq=X, y=ys, kernel=E.KERNEL_MATERN52, n_noise=1, n_mean=1, device=0)
        eng.factorize(bench.W.c4_natural(np.zeros(13)))
        dq, m = X.shape[1], b * q
        xd = torch.from_numpy(np.random.RandomState(0).rand(m, dq)).cuda()
        Ed = sobol_normal_samples(S, q, 0).cuda()
        Eh = Ed.cpu()
        vals = torch.empty(b, dtype=torch.float64, device="cuda")
        dx = torch.empty(m, dq, dtype=torch.float64, device="cuda")
        qmean = torch.empty(b, q, dtype=torch.float64, device="cuda")
        qcov = torch.empty(b, q, q, dtype=torch.float64, device="cuda")
        gm0 = torch.zeros(b, q, dtype=torch.float64, device="cuda")
        gc0 = torch.zeros(b, q, q, dtype=torch.float64, device="cuda")
        best_f = 0.5

        def fused():
            eng.acquisition_qbatch(xd, q, E.QACQ_EI, Ed, best_f=best_f, out_values=vals, out_d_xq=dx)

        def floor():
            eng.posterior_qbatch(xd, q, out_mean=qmean, out_cov=qcov)
            eng.posterior_qbatch_grad(xd, q, gm0, gc0, out=dx)

        def host():
            mean, cov = eng.posterior_qbatch(xd, q, out_mean=qmean, out_cov=qcov)
            mu = mean.cpu().requires_grad_(True)
            C = cov.cpu().requires_grad_(True)
            L = torch.linalg.cholesky(C)
            yv = mu[None] + torch.einsum("tij,sj->sti", L, Eh)
            v = (yv.max(-1).values - best_f).clamp_min(0).mean(0)
            g_mu, g_c = torch.autograd.grad(v.sum(), (mu, C))
            eng.posterior_qbatch_grad(xd, q, g_mu.cuda(), g_c.cuda(), out=dx)

        calls = (fused, floor, host)
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
        print("N=%5d b=%5d q=%3d S=%d: acquisition_qbatch %8.2f ms | posterior_qbatch + _grad %8.2f ms (%.2fx) | "
              "host MC path %8.2f ms (%.2fx)" % (n, b, q, S, a1, a2, a1 / a2, a3, a1 / a3), flush=True)
        tot, k = _kernel_ms(fused, "qacq_mc_kernel")
        print("    device ms of one acquisition_qbatch: total %.2f, qacq_mc_kernel %.3f" % (tot, k), flush=True)
        eng.close()
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
