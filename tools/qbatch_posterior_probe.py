"""Cost of the t-batch joint posterior: device-resident gpp_posterior_qbatch against gpp_predict, and
gpp_posterior_qbatch_grad against gpp_predict_grad, on the same b*q rows of the same engine (C4 workload, candidates,
upstream gradients and outputs on the GPU).

For each (N, b, q) the four calls alternate after a warm-up, and the medians of the repeats are printed with the two
ratios.  One call of each t-batch entry then runs under torch.profiler and the device time of its block kernels is
printed: the block-diagonal SYRK (qbatch_syrk_kernel) of the forward pass, and W = blockdiag(Gs) V
(qbatch_w_kernel), the in-batch K** term and the finish of the backward pass.  The card's name and power limit are
read in the same run.
Usage: python tools/qbatch_posterior_probe.py [--repeats R]
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

SIZES = ((512, 4096, 8), (2048, 1024, 32), (16384, 512, 8), (16384, 128, 128))
BLOCK_KERNELS = ("qbatch_syrk_kernel", "qbatch_w_kernel", "qbatch_inbatch_grad_kernel", "qbatch_grad_finish_kernel")


def _card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def _kernel_times(fn):
    """device milliseconds of one call: total, and per block kernel"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    tot = dict.fromkeys(BLOCK_KERNELS, 0.0)
    total = 0.0
    for ev in prof.events():
        if ev.device_type != torch.autograd.DeviceType.CUDA:
            continue
        total += ev.device_time / 1e3
        for k in BLOCK_KERNELS:
            if k in ev.name:
                tot[k] += ev.device_time / 1e3
    return total, tot


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=5)
    args = ap.parse_args()
    if E.device_count() < 1:
        raise SystemExit("qbatch_posterior_probe: no CUDA device visible")
    print("card: %s" % _card(), flush=True)
    for n, b, q in SIZES:
        X, y = bench.W.c4_workload(n)
        ys = (y - y.min()) / (y.max() - y.min())
        eng = E.Engine(xq=X, y=ys, kernel=E.KERNEL_MATERN52, n_noise=1, n_mean=1, device=0)
        eng.factorize(bench.W.c4_natural(np.zeros(13)))
        dq, m = X.shape[1], b * q
        xd = torch.from_numpy(np.random.RandomState(0).rand(m, dq)).cuda()
        gm = torch.from_numpy(np.random.RandomState(1).standard_normal((b, q))).cuda()
        gc = torch.from_numpy(np.random.RandomState(2).standard_normal((b, q, q))).cuda()
        mu, var = (torch.empty(m, dtype=torch.float64, device="cuda") for _ in range(2))
        dmu, dvar, dx = (torch.empty(m, dq, dtype=torch.float64, device="cuda") for _ in range(3))
        qmean = torch.empty(b, q, dtype=torch.float64, device="cuda")
        qcov = torch.empty(b, q, q, dtype=torch.float64, device="cuda")

        def plain():
            eng.predict(xd, out_mean=mu, out_var=var)

        def fwd():
            eng.posterior_qbatch(xd, q, out_mean=qmean, out_cov=qcov)

        def pgrad():
            eng.predict_grad(xd, out_mean=mu, out_var=var, out_d_mean=dmu, out_d_var=dvar)

        def bwd():
            eng.posterior_qbatch_grad(xd, q, gm, gc, out=dx)

        calls = (plain, fwd, pgrad, bwd)
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
        p, fw, pg, bw = (statistics.median(ts[f]) * 1e3 for f in calls)
        print("N=%5d b=%5d q=%3d (%d rows, dq=%d): predict %8.2f ms  posterior_qbatch %8.2f ms (%.2fx)  "
              "predict_grad %8.2f ms  posterior_qbatch_grad %8.2f ms (%.2fx)"
              % (n, b, q, m, dq, p, fw, fw / p, pg, bw, bw / pg), flush=True)
        ft, fk = _kernel_times(fwd)
        bt, bk = _kernel_times(bwd)
        print("    device ms: forward %.2f, block SYRK %.3f  |  backward %.2f, W %.3f, in-batch %.3f, finish %.3f"
              % (ft, fk["qbatch_syrk_kernel"], bt, bk["qbatch_w_kernel"], bk["qbatch_inbatch_grad_kernel"],
                 bk["qbatch_grad_finish_kernel"]), flush=True)
        eng.close()
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
