"""Cost of differentiable prediction: device-resident gpp_predict against gpp_predict_grad on the same engine.

For each (N, M) the two calls alternate after a warm-up of both, and the median of the repeats is printed with their
ratio and the effective FP64 rate of the triangular products over the whole call (predict: K* L^-T, M N^2 flop;
predict_grad: K* L^-T and U L^-1, 2 M N^2 flop).  --profile adds, per size, the device time of each kernel of one
predict_grad call (torch.profiler), to show where the time goes.  The card's name and power limit are read in the
same run.  Usage: python tools/predict_grad_probe.py [--repeats R] [--profile]
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

SIZES = ((512, 1 << 20), (2048, 1 << 18), (8192, 1 << 16), (16384, 8192))


def _card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--profile", action="store_true")
    args = ap.parse_args()
    if E.device_count() < 1:
        raise SystemExit("predict_grad_probe: no CUDA device visible")
    print("card: %s" % _card(), flush=True)
    for n, m in SIZES:
        X, y = bench.W.c4_workload(n)
        ys = (y - y.min()) / (y.max() - y.min())
        eng = E.Engine(xq=X, y=ys, kernel=E.KERNEL_MATERN52, n_noise=1, n_mean=1, device=0)
        eng.factorize(bench.W.c4_natural(np.zeros(13)))
        dq = X.shape[1]
        xd = torch.from_numpy(np.random.RandomState(0).rand(m, dq)).cuda()
        mu, var = (torch.empty(m, dtype=torch.float64, device="cuda") for _ in range(2))
        dm, dv = (torch.empty(m, dq, dtype=torch.float64, device="cuda") for _ in range(2))

        def plain():
            eng.predict(xd, out_mean=mu, out_var=var)

        def grad():
            eng.predict_grad(xd, out_mean=mu, out_var=var, out_d_mean=dm, out_d_var=dv)

        for f in (plain, grad, plain, grad):
            f()
        torch.cuda.synchronize()
        tp, tg = [], []
        for _ in range(args.repeats):
            for f, acc in ((plain, tp), (grad, tg)):
                t0 = time.perf_counter()
                f()
                torch.cuda.synchronize()
                acc.append(time.perf_counter() - t0)
        p, g = statistics.median(tp), statistics.median(tg)
        flop = float(m) * n * n
        print("N=%5d M=%7d dq=%d: predict %8.2f ms (%5.1f TFLOP/s)  predict_grad %8.2f ms (%5.1f TFLOP/s)  ratio %.2f"
              % (n, m, dq, p * 1e3, flop / p / 1e12, g * 1e3, 2 * flop / g / 1e12, g / p), flush=True)
        if args.profile:
            from torch.profiler import ProfilerActivity, profile
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                grad()
                torch.cuda.synchronize()
            tot = {}
            for ev in prof.events():
                if ev.device_type == torch.autograd.DeviceType.CUDA:
                    tot[ev.name] = tot.get(ev.name, 0.0) + ev.device_time / 1e3
            for name, ms in sorted(tot.items(), key=lambda kv: -kv[1])[:8]:
                print("    %8.2f ms  %s" % (ms, name[:110]), flush=True)
        eng.close()


if __name__ == "__main__":
    main()
