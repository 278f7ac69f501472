#!/bin/bash
# INT8-sliced vs DMMA at mid sizes (which arithmetic should be the default where), lazy panels on / off
mkdir -p gpurun_out
for n in 3072 4096 6144 8192 12288; do
for cfg in "1 0" "1 100000" "0 0"; do
  set -- $cfg
  GPP_OZ_LAZY_MIN=$2 python - <<PY 2>&1 | tail -1
import sys, time
sys.path[:0] = ['.', 'gp-plus_b200']
import numpy as np
import bench_workloads as W
from gpplus_b200 import _engine as E
n = $n
E.set_fp64_mode($1)
X, y = W.c4_workload(n)
ys = (y - y.min()) / (y.max() - y.min())
eng = E.Engine(xq=X, y=ys, kernel=E.KERNEL_MATERN52, n_noise=1, n_mean=1, device=0)
th = W.c4_theta_points(W.c4_model(256))
outs = []
for k in range(6):
    o = eng.mll_grad(W.c4_natural(th[1 + k % 2]), want_grad=True)
    t = eng.timings()
    if k >= 2: outs.append(t)
tot = np.median([t['total'] for t in outs])
print("n=%5d fp64_mode %d lazy_min $2: total %.3f ms  chol %.3f trtri %.3f lauum %.3f  nll %.12e" % (n, eng.fp64_mode(), tot, outs[-1]['cholesky'], outs[-1]['trtri'], outs[-1]['lauum'], o['nll']))
eng.close()
PY
done
done
