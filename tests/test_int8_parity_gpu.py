"""Parity of the INT8-sliced FP64 path (csrc/oz_gemm.cuh, oz_split.cuh, oz_chol.cuh) against the CPU oracle at the
shapes and models it serves, and against the exact-DMMA arithmetic on the same settings.

Every case runs on a handle that reports fp64_mode() == FP64_INT8 and checks what the DMMA-arm parity tests check
(test_engine_gpu.check_case), at the same tolerances: covariance 1e-12 of max|K|, nll 1e-9 relative, every gradient
1e-8 of its max-norm, equal jitter, predictions with and without noise 1e-9.  The cross-arm check re-runs the problem
with gpp_set_fp64_mode(FP64_DMMA): nll within 1e-11 relative, L^-1 and K^-1 within 1e-12 of their largest entry.
For that comparison to be meaningful at the FP64 rounding level the cases keep kappa(K_y) <= 1e4 (checked here).

Cases (T = Np / 128 tiles): the default switch point T = 23 / 24 (N = 2944, 2945; 2945 has 127 padded rows); RBF with
a 2-d latent map over 25 levels, 4 noise groups and 4 means with a zero-mean group (N = 3073: the inverse level
hb = 8 has a 1-tile last group); Matern-3/2 with 3 latent passes (N = 6001: ragged last groups at hb = 4, 8, 32); lazy
panels of 2, 12 and 16 tiles (last panels of 1, 1 and 9 tiles); the forced INT8 arithmetic with the smallest stage
thresholds at N = 1100 and 2300; the jitter ladder and error mapping; acquisition scores from an INT8 factorisation;
and N = 17600 (T = 138: two K^-1 segments, plane buffers above 2^31 bytes) against the committed oracle output.
"""
import json
import os

import numpy as np
import pytest
import scipy.sparse.linalg as sla

import bench_workloads as W
from oracle import gp_oracle as O
from problems import engine_kwargs, make_candidates, make_hyper, make_problem

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
NLL_RTOL, GRAD_RTOL, K_RTOL, PRED_TOL = 1e-9, 1e-8, 1e-12, 1e-9
ARM_NLL_RTOL, ARM_INV_RTOL = 1e-11, 1e-12
KAPPA_MAX = 1e4

_oracle_cache = {}


def rel(a, b):
    a, b = np.asarray(a, dtype=float), np.asarray(b, dtype=float)
    return float(np.max(np.abs(a - b)) / max(1e-300, np.max(np.abs(b))))


def _oracle(key, p, h):
    if key not in _oracle_cache:
        _oracle_cache[key] = O.mll(p, h, want_grad=True, return_mats=True)
    return _oracle_cache[key]


def _noise_diag(p, h):
    noise = np.asarray(h["noise"], dtype=float)
    return noise[p["noise_idx"]] if p["noise_idx"] is not None else np.full(p["n"], noise[0])


def _kappa_bound(p, h, K):
    """Upper bound of kappa(K_y), K_y = K + diag(noise): K is positive semi-definite, so lambda_min(K_y) >= min noise."""
    d = _noise_diag(p, h)
    lam = float(sla.eigsh(K, k=1, which="LA", tol=1e-8, return_eigenvectors=False)[0])
    return (lam * (1.0 + 1e-6) + d.max()) / d.min()


def _env(monkeypatch, env):
    for k, v in (env or {}).items():
        monkeypatch.setenv(k, v)


def check_int8_case(name, p, h, monkeypatch, env=None, mode=-1, cand=48):
    """Full oracle check on the INT8 arm (mode: -1 = by size, or FP64_INT8 forced) and the cross-arm check."""
    from gpplus_b200 import _engine as E
    _env(monkeypatch, env)
    ref = _oracle(name.split("/")[0], p, h)
    kappa = _kappa_bound(p, h, ref["K"])
    assert kappa <= KAPPA_MAX, (name, kappa)
    errs, bounds = {}, {}

    def record(key, err, bound):
        errs[key], bounds[key] = err, bound

    prev = E.set_fp64_mode(mode)
    try:
        eng = E.Engine(**engine_kwargs(p))
        try:
            assert eng.fp64_mode() == E.FP64_INT8, name
            record("K", rel(eng.covariance(h), ref["K"]), K_RTOL)
            out = eng.mll_grad(h, want_grad=True)
            record("nll", abs(out["nll"] - ref["nll"]) / abs(ref["nll"]), NLL_RTOL)
            assert out["jitter"] == ref["jitter"], name
            for k in ("d_w", "d_noise", "d_z", "d_beta"):
                if k in ref and np.size(ref[k]):
                    record(k, rel(out[k], ref[k]), GRAD_RTOL)
            record("d_sigma_f2", abs(out["d_sigma_f2"] - ref["d_sigma_f2"]) / max(1.0, abs(ref["d_sigma_f2"])), GRAD_RTOL)
            li, ki = eng.fetch("Linv"), eng.fetch("Kinv")
            val = eng.mll_grad(h, want_grad=False)
            assert val["nll"] == out["nll"], name   # value-only path: bit-identical value
            c = make_candidates(p, cand)
            for inc in (False, True):
                mu_ref, var_ref = O.predict(p, h, c, include_noise=inc)
                mu, var = eng.predict(c["xq"], c["level_idx"], c["noise_idx"], c["mean_idx"], include_noise=inc)
                record("mu%d" % inc, np.max(np.abs(mu - mu_ref)) / max(1.0, np.max(np.abs(mu_ref))), PRED_TOL)
                record("var%d" % inc, np.max(np.abs(var - var_ref)) / max(1.0, np.max(np.abs(var_ref))), PRED_TOL)
        finally:
            eng.close()
        E.set_fp64_mode(E.FP64_DMMA)
        eng = E.Engine(**engine_kwargs(p))
        try:
            assert eng.fp64_mode() == E.FP64_DMMA, name
            dm = eng.mll_grad(h, want_grad=True)
            record("arm_nll", abs(out["nll"] - dm["nll"]) / abs(dm["nll"]), ARM_NLL_RTOL)
            record("arm_Linv", rel(li, eng.fetch("Linv")), ARM_INV_RTOL)
            record("arm_Kinv", rel(ki, eng.fetch("Kinv")), ARM_INV_RTOL)
        finally:
            eng.close()
    finally:
        E.set_fp64_mode(prev)
    print("INT8 parity %s (kappa <= %.0f): %s" % (name, kappa, ", ".join("%s %.2e (%.0e)" % (k, errs[k], bounds[k])
                                                                        for k in errs)))
    bad = [k for k in errs if not errs[k] <= bounds[k]]
    assert not bad, (name, {k: (errs[k], bounds[k]) for k in bad})


def _multi_problem():
    p = make_problem(3073, 10, 0, dz=2, n_combo=25, n_noise=4, n_mean=4, seed=301, zero_mean_group=True)
    return p, make_hyper(p, seed=302, noise=0.05)


@pytest.mark.parametrize("n", [2944, 2945])
def test_default_switch_point(n, monkeypatch):
    """T = 23 stays on DMMA by default and T = 24 switches to INT8 (csrc/engine.cu read_config); 2944 is checked with
    the INT8 arithmetic forced."""
    from gpplus_b200 import _engine as E
    p = make_problem(n, 10, 2, seed=310 + n)
    h = make_hyper(p, seed=311, noise=0.05)
    prev = E.set_fp64_mode(-1)
    try:
        eng = E.Engine(**engine_kwargs(p))
        try:
            assert eng.fp64_mode() == (E.FP64_INT8 if n == 2945 else E.FP64_DMMA)
        finally:
            eng.close()
    finally:
        E.set_fp64_mode(prev)
    check_int8_case("switch%d" % n, p, h, monkeypatch, mode=-1 if n == 2945 else E.FP64_INT8)


def test_latent_map_multi_noise_multi_mean_rbf(monkeypatch):
    p, h = _multi_problem()
    check_int8_case("multi", p, h, monkeypatch)


def test_multi_pass_matern32(monkeypatch):
    p = make_problem(6001, 10, 1, dz=2, n_combo=9, n_noise=2, n_mean=2, seed=320, n_pass=3)
    h = make_hyper(p, seed=321, noise=0.05)
    check_int8_case("npass3", p, h, monkeypatch, cand=32)


@pytest.mark.parametrize("pb", ["2", "12", "16"])
def test_lazy_panels_with_short_last_panel(pb, monkeypatch):
    p, h = _multi_problem()
    check_int8_case("multi/lazy%s" % pb, p, h, monkeypatch, env={"GPP_OZ_LAZY_MIN": "24", "GPP_OZ_LAZY_PB": pb})


@pytest.mark.parametrize("n", [1100, 2300])
def test_forced_int8_with_smallest_stage_thresholds(n, monkeypatch):
    """Forced INT8 (T >= 8) with every trailing update (oz_use_trailing: T - c0 >= 1) and every inverse level
    (oz_use_level: hb >= 1) on the integer GEMM."""
    from gpplus_b200 import _engine as E
    p = make_problem(n, 10, 2, dz=1, n_combo=6, n_noise=2, seed=330 + n)
    h = make_hyper(p, seed=331, noise=0.05)
    check_int8_case("forced%d" % n, p, h, monkeypatch, env={"GPP_OZ_MIN_TRAIL": "1", "GPP_OZ_MIN_LEVEL": "1"},
                    mode=E.FP64_INT8)


def test_jitter_ladder_and_error_mapping():
    """K_y = K - (lambda_min(K) + 5e-7) I: the rungs 0, 1e-8 and 1e-7 fail and 1e-6 succeeds, each by a margin of at
    least 100 x the rounding level N eps lambda_max(K_y) (asserted from the oracle's eigenvalues)."""
    from gpplus_b200 import _engine as E
    p = make_problem(3073, 10, 2, seed=340)
    h = make_hyper(p, seed=341, noise=0.05)
    K = O.mll(p, h, want_grad=False, return_mats=True)["K"]
    lam = np.linalg.eigvalsh(K)
    h["noise"] = np.array([-(lam[0] + 5e-7)])
    lam_y = lam + h["noise"][0]
    rounding = p["n"] * np.finfo(float).eps * lam_y[-1]
    for jit in (0.0, 1e-8, 1e-7, 1e-6):
        assert abs(lam_y[0] + jit) >= 100.0 * rounding, (jit, lam_y[0] + jit, rounding)
    ref = O.mll(p, h, want_grad=False)
    assert ref["jitter"] == 1e-6
    eng = E.Engine(**engine_kwargs(p))
    try:
        assert eng.fp64_mode() == E.FP64_INT8
        out = eng.mll_grad(h, want_grad=True)
        assert out["jitter"] == ref["jitter"]
        # kappa(K_y + 1e-6 I) ~ lambda_max / 5e-7: the objective is only good to about kappa eps here
        assert abs(out["nll"] - ref["nll"]) <= 1e-6 * abs(ref["nll"]), (out["nll"], ref["nll"])
        hn = dict(h)
        hn["sigma_f2"] = -1.0
        with pytest.raises(E.NotPSDError):
            eng.mll_grad(hn, want_grad=True)
        hn["sigma_f2"] = float("nan")
        with pytest.raises(E.NanError):
            eng.mll_grad(hn, want_grad=True)
        out = eng.mll_grad(make_hyper(p, seed=342, noise=0.05), want_grad=True)
        assert np.isfinite(out["nll"])
    finally:
        eng.close()


def test_acquisition_scores_from_an_int8_factorisation():
    from gpplus_b200 import _engine as E
    p = make_problem(3073, 8, 0, dz=2, n_combo=5, n_noise=5, n_mean=1, seed=350)
    h = make_hyper(p, seed=351, noise=0.05)
    c = make_candidates(p, 5000, seed=352)
    src = c["level_idx"].astype(np.int32)
    cost = np.array([1000.0, 100.0, 10.0, 100.0, 10.0])
    kinds = [E.ACQ_HF, E.ACQ_LF, E.ACQ_LF, E.ACQ_LF, E.ACQ_EI]
    best_f = np.array([0.4, 0.5, 0.6, 0.5, 0.45])
    mu, var = O.predict(p, h, c, include_noise=False)
    mean, std = 2.0 + 3.0 * mu, np.sqrt(var) * 3.0
    eng = E.Engine(**engine_kwargs(p))
    try:
        assert eng.fp64_mode() == E.FP64_INT8
        eng.factorize(h)
        for maximize in (True, False):
            s, i, scores = eng.acq_argmax(c["xq"], src, cost, kinds, best_f, level_idx=c["level_idx"],
                                          maximize=maximize, y_min=2.0, y_std=3.0, return_scores=True)
            want = np.empty(c["m"])
            for k in range(5):
                sel = src == k
                want[sel] = O.acquisition(mean[sel], std[sel], kinds[k], best_f[k], cost[k] * np.ones(sel.sum()),
                                          maximize=maximize)
            err = np.max(np.abs(scores - want)) / max(1.0, np.max(np.abs(want)))
            print("INT8 acquisition maximize=%s: scores %.2e (bound 1e-9)" % (maximize, err))
            assert err < 1e-9
            assert i == int(np.argmax(want)) and s == scores[i]
    finally:
        eng.close()


def _check_against(out, ref, where):
    assert abs(out["nll"] - ref["nll"]) <= NLL_RTOL * abs(ref["nll"]), (where, out["nll"], ref["nll"])
    assert out["jitter"] == ref["jitter"], (where, out["jitter"], ref["jitter"])
    g = np.concatenate([out["d_w"], [out["d_sigma_f2"]], out["d_noise"], out["d_beta"]])
    gr = np.concatenate([np.asarray(ref["d_w"]), [ref["d_sigma_f2"]], np.asarray(ref["d_noise"]),
                         np.asarray(ref["d_beta"])])
    err = np.max(np.abs(g - gr)) / np.max(np.abs(gr))
    assert err <= GRAD_RTOL, (where, err)
    return abs(out["nll"] - ref["nll"]) / abs(ref["nll"]), err, out["nll"], g


def test_beyond_the_headline_n17600():
    """T = 138 > 128: K^-1 in two K segments, a top inverse level with a 10-tile last group, a last lazy panel of
    6 tiles, 7 Np^2 > 2^31 bytes per plane buffer.  Against tests/golden/c4_n17600_matern52.json (generated with
    python tests/golden/make_golden.py --c4 17600) and against the DMMA arm."""
    from gpplus_b200 import _engine as E
    n = 17600
    gold = json.load(open(os.path.join(HERE, "golden", "c4_n17600_matern52.json")))
    assert gold["n"] == n
    thetas = W.c4_theta_points(W.c4_model(256))
    X, y = W.c4_workload(n)
    ys = (y - y.min()) / (y.max() - y.min())
    outs = {}
    prev = E.set_fp64_mode(-1)
    try:
        for mode in (-1, E.FP64_DMMA):
            E.set_fp64_mode(mode)
            eng = E.Engine(xq=X, y=ys, kernel=E.KERNEL_MATERN52, n_noise=1, n_mean=1, device=0)
            try:
                assert eng.fp64_mode() == (E.FP64_INT8 if mode == -1 else E.FP64_DMMA)
                for pt in gold["points"]:
                    np.testing.assert_array_equal(np.asarray(pt["theta"]), thetas[pt["index"]])
                    out = eng.mll_grad(W.c4_natural(thetas[pt["index"]]), want_grad=True)
                    outs[(mode, pt["index"])] = _check_against(out, pt, "n=17600 mode %d point %d" % (mode, pt["index"]))
            finally:
                eng.close()
    finally:
        E.set_fp64_mode(prev)
    for pt in gold["points"]:
        (e8, g8, nll8, a), (ed, gd, nlld, b) = outs[(-1, pt["index"])], outs[(E.FP64_DMMA, pt["index"])]
        arm_nll = abs(nll8 - nlld) / abs(nlld)
        arm = np.max(np.abs(a - b)) / np.max(np.abs(b))
        print("INT8 n=17600 point %d: nll %.2e grad %.2e vs oracle (DMMA arm: %.2e, %.2e); cross-arm nll %.2e "
              "(bound 1e-11) grad %.2e (bound 1e-10)" % (pt["index"], e8, g8, ed, gd, arm_nll, arm))
        assert arm_nll <= ARM_NLL_RTOL and arm <= 1e-10, (pt["index"], arm_nll, arm)
