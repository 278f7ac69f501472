"""Cost of the one-shot knowledge gradient with input gradients (gpp_kg_qbatch) on the C4 workload, device-resident,
against Monte-Carlo qEI with S = 512 samples and the gradient (gpp_acq_qbatch) at the same (N, b, q_tot): both share
the t-batch posterior and its backward, and differ only in the per-t-batch kernel.  The two arms alternate after a
warm-up and the medians of the repeats are printed.  One call of each then runs under torch.profiler and the device
time of kg_block_kernel and of qacq_mc_kernel is printed.  The card's name and power limit are read in the same run.
Usage: python tools/kg_probe.py [--repeats R]
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

SIZES = ((512, 1024, 4, 60), (2048, 256, 4, 60), (16384, 64, 4, 124))  # (N, b, q, F)
S = 512


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
        raise SystemExit("kg_probe: no CUDA device visible")
    print("card: %s" % _card(), flush=True)
    for n, b, q, nf in SIZES:
        q_tot = q + nf
        X, y = bench.W.c4_workload(n)
        ys = (y - y.min()) / (y.max() - y.min())
        eng = E.Engine(xq=X, y=ys, kernel=E.KERNEL_MATERN52, n_noise=1, n_mean=1, device=0)
        eng.factorize(bench.W.c4_natural(np.zeros(13)))
        dq, m = X.shape[1], b * q_tot
        xd = torch.from_numpy(np.random.RandomState(0).rand(m, dq)).cuda()
        Ek = sobol_normal_samples(nf, q, 0).cuda()
        Ea = sobol_normal_samples(S, q_tot, 0).cuda()
        vals = torch.empty(b, dtype=torch.float64, device="cuda")
        dx = torch.empty(m, dq, dtype=torch.float64, device="cuda")

        def kg():
            eng.kg_qbatch(xd, q, nf, Ek, out_values=vals, out_d_xq=dx)

        def qei():
            eng.acquisition_qbatch(xd, q_tot, E.QACQ_EI, Ea, best_f=0.5, out_values=vals, out_d_xq=dx)

        calls = (kg, qei)
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
        a1, a2 = (statistics.median(ts[f]) * 1e3 for f in calls)
        print("N=%5d b=%5d q_tot=%d+%d: kg_qbatch %8.2f ms | acquisition_qbatch qEI S=%d %8.2f ms (kg/qEI %.2fx)"
              % (n, b, q, nf, a1, S, a2, a1 / a2), flush=True)
        tk, k = _kernel_ms(kg, "kg_block_kernel")
        ta, ka = _kernel_ms(qei, "qacq_mc_kernel")
        print("    device ms of one call: kg_qbatch total %.2f, kg_block_kernel %.3f | acquisition_qbatch total %.2f, "
              "qacq_mc_kernel %.3f" % (tk, k, ta, ka), flush=True)
        eng.close()
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
