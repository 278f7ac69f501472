"""gpp_predict_grad on the B200: derivatives of the predictive mean / variance w.r.t. the candidates' quantitative
inputs against torch autograd through the dense CPU oracle (tests/predict_grad_reference.py), bitwise agreement of mean / variance with gpp_predict,
determinism, and GP_Plus.predict_with_grad end to end."""
import numpy as np
import pytest
import torch
from scipy.optimize import minimize

from problems import engine_kwargs, make_candidates, make_hyper, make_problem

pytestmark = pytest.mark.gpu

# worst errors relative to the batch's max-norm observed on one B200 (1000 W power limit): d_mean 3.9e-10 and d_var
# 3.2e-11 with the INT8-sliced factor at N = 3200, at most 2.7e-12 / 1.0e-12 on every DMMA case
D_MEAN_TOL = 2e-9
D_VAR_TOL = 2e-10


def _rel(a, b):
    return float(np.max(np.abs(a - b)) / max(1e-300, np.max(np.abs(b)))) if b.size else 0.0


def _check(p, h, c, include_noise=False, mode="expansion", fp64=None):
    from gpplus_b200 import _engine as E
    from predict_grad_reference import predict_grad as reference_predict_grad
    prev = E.set_fp64_mode(fp64) if fp64 is not None else None
    try:
        eng = E.Engine(**engine_kwargs(p))
    finally:
        if fp64 is not None:
            E.set_fp64_mode(prev)
    try:
        if fp64 is not None:
            assert eng.fp64_mode() == fp64
        eng.factorize(h)
        kw = dict(level_idx=c["level_idx"], noise_idx=c["noise_idx"], mean_idx=c["mean_idx"],
                  include_noise=include_noise)
        mu, var, dm, dv = eng.predict_grad(c["xq"], **kw)
        mu0, var0 = eng.predict(c["xq"], **kw)
        assert np.array_equal(mu, mu0) and np.array_equal(var, var0)
        again = eng.predict_grad(c["xq"], **kw)
        assert all(np.array_equal(a, b) for a, b in zip((mu, var, dm, dv), again))
    finally:
        eng.close()
    rmu, rvar, rdm, rdv = reference_predict_grad(p, h, c, include_noise, mode=mode)
    assert dm.shape == (c["m"], p["dq"]) and dv.shape == (c["m"], p["dq"])
    assert np.all(np.isfinite(dm)) and np.all(np.isfinite(dv))
    errs = (_rel(dm, rdm), _rel(dv, rdv))
    print("d_mean %.2e d_var %.2e" % errs)
    assert errs[0] <= D_MEAN_TOL and errs[1] <= D_VAR_TOL, errs
    return dm, dv


@pytest.mark.parametrize("kernel", [0, 1, 2])
@pytest.mark.parametrize("n", [1, 127, 129, 300])
def test_gradients_match_oracle(kernel, n):
    p = make_problem(n, 4, kernel, seed=n + kernel)
    _check(p, make_hyper(p, seed=3), make_candidates(p, 300, seed=5))


@pytest.mark.parametrize("n_pass", [1, 3])
def test_latent_map_and_ensemble(n_pass):
    p = make_problem(260, 3, 2, dz=2, n_combo=6, n_pass=n_pass, seed=11)
    _check(p, make_hyper(p, seed=4), make_candidates(p, 200, seed=6))


def test_noise_groups_and_means_with_zero_mean_group():
    p = make_problem(300, 5, 0, dz=2, n_combo=4, n_noise=3, n_mean=3, zero_mean_group=True, seed=12)
    c = make_candidates(p, 257, seed=7)
    assert c["mean_idx"].min() == -1
    _check(p, make_hyper(p, seed=5, noise=1e-2), c, include_noise=True)


def test_widest_input():
    p = make_problem(400, 32, 1, seed=13)
    _check(p, make_hyper(p, seed=6, w_scale=0.02), make_candidates(p, 150, seed=8))


def test_no_quantitative_input_gives_empty_gradients():
    p = make_problem(200, 0, 0, dz=2, n_combo=5, seed=14)
    dm, dv = _check(p, make_hyper(p, seed=7), make_candidates(p, 64, seed=9))
    assert dm.shape == (64, 0) and dv.shape == (64, 0)


@pytest.mark.parametrize("fp64", ["dmma", "int8"])
def test_int8_sliced_factor(fp64):
    from gpplus_b200 import _engine as E
    p = make_problem(3200, 4, 2, seed=15)
    _check(p, make_hyper(p, seed=8, noise=1e-3), make_candidates(p, 300, seed=10),
           fp64=E.FP64_DMMA if fp64 == "dmma" else E.FP64_INT8)


@pytest.mark.parametrize("kernel", [1, 2])
def test_candidates_on_training_points(kernel):
    p = make_problem(200, 3, kernel, seed=16)
    c = {"m": 50, "xq": p["xq"][:50].copy(), "level_idx": None, "noise_idx": None, "mean_idx": None}
    _check(p, make_hyper(p, seed=9), c, mode="direct")


@pytest.mark.parametrize("dq", [4, 32])
def test_chunking_is_invisible(dq):
    """Mean / variance equal gpp_predict's and gradients do not depend on the chunk across a chunk boundary
    (np = 16512: the prediction chunk holds 8064 candidates; at dq = 32 this path's chunk shrinks to 3968)."""
    from gpplus_b200 import _engine as E
    p = make_problem(16500, dq, 0, seed=29)
    h = make_hyper(p, seed=14, noise=1e-2, w_scale=0.3 if dq == 4 else 0.02)
    c = make_candidates(p, 9000, seed=4)
    eng = E.Engine(**engine_kwargs(p))
    try:
        eng.factorize(h)
        mu, var, dm, dv = eng.predict_grad(c["xq"])
        mu0, var0 = eng.predict(c["xq"])
        assert np.array_equal(mu, mu0) and np.array_equal(var, var0)
        for lo, hi in ((3900, 4100), (7990, 8100)):
            part = eng.predict_grad(c["xq"][lo:hi])
            assert all(np.array_equal(a[lo:hi], b) for a, b in zip((mu, var, dm, dv), part))
        assert np.all(np.isfinite(dm)) and np.all(np.isfinite(dv)) and np.count_nonzero(dm) > 0
    finally:
        eng.close()


def _models():
    import test_model_gpu as TM
    return [("c1", TM._c1), ("c2_matern52", lambda: TM._c2("Matern52Kernel")), ("c3", TM._c3)]


@pytest.mark.parametrize("name", ["c1", "c2_matern52", "c3"])
def test_predict_with_grad_on_models(name):
    m, _, Xte, _ = dict(_models())[name]()
    Xq = Xte[:8].clone()
    x = Xq.clone().requires_grad_(True)
    mean, std = m.predict_with_grad(x, return_std=True, include_noise=True)
    mean0, std0 = m.predict(Xq, return_std=True, include_noise=True)
    assert torch.equal(mean.detach(), mean0) and torch.equal(std.detach(), std0)
    g_mean, = torch.autograd.grad(mean.sum(), x, retain_graph=True)
    g_std, = torch.autograd.grad(std.sum(), x)
    cols = m._quant_columns()
    other = [k for k in range(Xq.shape[1]) if k not in cols]
    assert len(other) == {"c1": 0, "c2_matern52": 2, "c3": 1}[name]
    assert torch.count_nonzero(g_mean[:, other]) == 0 and torch.count_nonzero(g_std[:, other]) == 0
    # the variance (sf2 minus a sum of squares) carries rounding of order 1e-16 sf2, which the difference quotient
    # divides by the step: at 1e-6 the c3 std differences came out 3.8e-6 off the analytic gradient
    eps = 1e-5
    fd_m, fd_s = torch.zeros_like(Xq), torch.zeros_like(Xq)
    for d in cols:
        e = torch.zeros_like(Xq)
        e[:, d] = eps
        mp, sp = m.predict(Xq + e, return_std=True, include_noise=True)
        mm, sm = m.predict(Xq - e, return_std=True, include_noise=True)
        fd_m[:, d], fd_s[:, d] = (mp - mm) / (2 * eps), (sp - sm) / (2 * eps)
    err_m = float((g_mean - fd_m).abs().max() / fd_m.abs().max())
    err_s = float((g_std - fd_s).abs().max() / fd_s.abs().max())
    print("%s: central differences vs autograd: mean %.2e std %.2e" % (name, err_m, err_s))
    assert err_m <= 1e-6 and err_s <= 1e-6


def test_lbfgsb_with_analytic_gradient_reaches_the_finite_difference_optimum():
    """Maximise AF_HF_Engineering over the inputs of a borehole model with scipy L-BFGS-B, once with jac=True from
    predict_with_grad and once with scipy's finite differences over predict(), from the same start."""
    import test_model_gpu as TM
    from gpplus_b200.bayesian_optimizations.AFs import AF_HF_Engineering
    m, _, Xte, yte = TM._c1()
    best_f = float(yte.max())
    d = Xte.shape[1]
    cost = lambda s: 1.0  # noqa: E731

    def neg_af(x, grad):
        xt = torch.tensor(x.reshape(1, d), dtype=torch.float64, requires_grad=grad)
        if grad:
            mean, std = m.predict_with_grad(xt, return_std=True, include_noise=True)
        else:
            mean, std = m.predict(xt, return_std=True, include_noise=True)
        f = -AF_HF_Engineering(best_f, mean.reshape(-1, 1), std.reshape(-1, 1), xt.detach(), cost).sum()
        if not grad:
            return float(f)
        g, = torch.autograd.grad(f, xt)
        return float(f), g.numpy().reshape(-1)

    x0 = Xte[0].numpy().copy()
    bounds = [(0.0, 1.0)] * d
    opts = {"ftol": 1e-12, "gtol": 1e-8}
    ana = minimize(neg_af, x0, args=(True,), jac=True, method="L-BFGS-B", bounds=bounds, options=opts)
    fd = minimize(neg_af, x0, args=(False,), method="L-BFGS-B", bounds=bounds, options=opts)
    print("analytic: f %.10f nfev %d; finite differences: f %.10f nfev %d" % (ana.fun, ana.nfev, fd.fun, fd.nfev))
    assert ana.success and ana.fun < neg_af(x0, False)
    assert abs(ana.fun - fd.fun) <= 1e-6 * max(1.0, abs(fd.fun))
    assert np.max(np.abs(ana.x - fd.x)) <= 1e-3
