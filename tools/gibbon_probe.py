"""Cost of GIBBON (gpp_gibbon_qbatch) on the C4 workload (N = 16384), device-resident: values-only and gradient calls at
b = 512 for q in {1, 4} and projected 0 / 1, against the one-shot knowledge gradient with the gradient
(gpp_kg_qbatch) at q = 1, F = 64 in the same process, and gpp_max_value_quartiles over m = 2^20 candidates.  Every
call is warmed up, the arms alternate and the medians of the repeats are printed.  One gradient call of GIBBON and
of KG then runs under torch.profiler and the device time of gibbon_block_kernel and kg_block_kernel is printed.  The
card's name and power limit are read in the same run.
Usage: python tools/gibbon_probe.py [--repeats R] [--n N]
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

B, K, M_QUART = 512, 10, 1 << 20


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
    ap.add_argument("--n", type=int, default=16384)
    args = ap.parse_args()
    if E.device_count() < 1:
        raise SystemExit("gibbon_probe: no CUDA device visible")
    print("card: %s" % _card(), flush=True)
    n = args.n
    X, y = bench.W.c4_workload(n)
    ys = (y - y.min()) / (y.max() - y.min())
    eng = E.Engine(xq=X, y=ys, kernel=E.KERNEL_MATERN52, n_noise=1, n_mean=1, device=0)
    eng.factorize(bench.W.c4_natural(np.zeros(13)))
    dq = X.shape[1]
    rng = np.random.RandomState(0)
    mv = torch.from_numpy(1.0 + 0.1 * np.abs(rng.standard_normal(K))).cuda()
    vals = torch.empty(B, dtype=torch.float64, device="cuda")
    arms = []
    for q in (1, 4):
        for proj in (False, True):
            m = B * q * (2 if proj else 1)
            xd = torch.from_numpy(rng.rand(m, dq)).cuda()
            dx = torch.empty(m, dq, dtype=torch.float64, device="cuda")
            for grad in (False, True):
                def call(xd=xd, dx=dx, q=q, proj=proj, grad=grad):
                    eng.gibbon_qbatch(xd, q, mv, projected=proj, want_grad=grad, out_values=vals,
                                      out_d_xq=dx if grad else None)
                arms.append(("gibbon_qbatch q=%d projected=%d %s" % (q, proj, "grad  " if grad else "values"), call))
    nf = 64
    xk = torch.from_numpy(rng.rand(B * (1 + nf), dq)).cuda()
    dk = torch.empty(B * (1 + nf), dq, dtype=torch.float64, device="cuda")
    ek = sobol_normal_samples(nf, 1, 0).cuda()

    def kg():
        eng.kg_qbatch(xk, 1, nf, ek, out_values=vals, out_d_xq=dk)

    arms.append(("kg_qbatch q=1 F=64 grad", kg))
    xm = torch.from_numpy(rng.rand(M_QUART, dq)).cuda()
    qout = torch.empty(3, dtype=torch.float64, device="cuda")

    def quart():
        eng.max_value_quartiles(xm, out=qout)

    arms.append(("max_value_quartiles m=2^20", quart))
    for _, f in arms:
        f()
    torch.cuda.synchronize()
    ts = {name: [] for name, _ in arms}
    for _ in range(args.repeats):
        for name, f in arms:
            t0 = time.perf_counter()
            f()
            torch.cuda.synchronize()
            ts[name].append(time.perf_counter() - t0)
    print("N=%d b=%d K=%d, medians of %d:" % (n, B, K, args.repeats), flush=True)
    for name, _ in arms:
        print("  %-40s %9.2f ms" % (name, statistics.median(ts[name]) * 1e3), flush=True)
    g = [f for name, f in arms if name.startswith("gibbon_qbatch q=1 projected=1 grad")][0]
    tg, kgk = _kernel_ms(g, "gibbon_block_kernel")
    tk, kk = _kernel_ms(kg, "kg_block_kernel")
    print("device ms of one call: gibbon_qbatch q=1 projected=1 grad total %.2f, gibbon_block_kernel %.3f | "
          "kg_qbatch total %.2f, kg_block_kernel %.3f" % (tg, kgk, tk, kk), flush=True)
    eng.close()


if __name__ == "__main__":
    main()
