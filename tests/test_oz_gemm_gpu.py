"""The INT8-sliced FP64 GEMM (csrc/oz_gemm.cuh, csrc/oz_split.cuh) below the engine, through tools/oz_lab.cu:

* digit planes of the split kernels against a host re-computation (bit-exact; representation error <= 2^-56 of the row scale),
  transposed split against the row split (bit-exact);
* the tcgen05 integer GEMM against the exact host sum over the 28 plane pairs (<= 1e-15 of sum |a||b|) and against a
  long-double product;
* alpha / beta / K sub-range, the lower-triangular K-range map (K^-1 = M^T M shape) and the batched KSEL_TJ form of the
  inverse levels against the DMMA kernel;
* check groups, one test each, against long-double or int64 host products (see tools/oz_lab.cu): the ragged batched
  inverse levels, the filtered / lazy-panel tile maps, K ranges accumulated in segments, int32 accumulator limits with
  digit planes written directly, and the split of rows with extreme exponents (2^-1074 .. 2^996, NaN / Inf rows).

The binary is built here with nvcc when it is missing or older than its sources (the GPU box has the same toolchain).
"""
import os
import shutil
import subprocess

import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "tools", "oz_lab")
SRC = [os.path.join(ROOT, "tools", "oz_lab.cu")] + [os.path.join(ROOT, "gp-plus_b200", "csrc", f) for f in
                                                     ("oz_gemm.cuh", "oz_split.cuh", "oz_chol.cuh", "dgemm_dmma.cuh",
                                                                          "tma.cuh")]


def _build():
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    stale = (not os.path.exists(EXE)) or any(os.path.getmtime(s) > os.path.getmtime(EXE) for s in SRC)
    if stale:
        subprocess.check_call([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo",
                               "-o", EXE, SRC[0]])


def test_int8_sliced_gemm_checks():
    _build()
    r = subprocess.run([EXE, "check"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "check: ok" in r.stdout, r.stdout[-2000:]
    assert "digit mismatches 0" in r.stdout and "mismatches against split_rows 0" in r.stdout, r.stdout[-2000:]


@pytest.mark.parametrize("group", ["ragged", "maps", "segments", "limits", "exponents"])
def test_int8_sliced_check_groups(group):
    _build()
    r = subprocess.run([EXE, group], capture_output=True, text=True, timeout=600)
    print(r.stdout)
    assert r.returncode == 0 and "%s: ok" % group in r.stdout, r.stdout[-3000:] + r.stderr[-2000:]


def test_int8_rate_probe_through_the_c_abi():
    from gpplus_b200 import _engine as E
    t256 = E.probe_i8(256, 2048)
    t128 = E.probe_i8(128, 2048)
    t64 = E.probe_i8(64, 2048)
    # nominal dense INT8 peak 4500 TOP/s; N = 64 is limited by shared-memory operand reads (6 KB per MMA at 128 B/clk)
    assert 3000.0 < t256 < 5200.0, t256
    assert 0.85 * t256 < t128 < 1.05 * t256, (t128, t256)
    assert 0.5 * t256 < t64 < 0.8 * t256, (t64, t256)
