"""One-shot knowledge gradient (qKG): the CPU reference against botorch's refit semantics and central differences, and
the host side (GPR.knowledge_gradient, the autograd Function behind it, optimize_knowledge_gradient and
optimize_posterior_mean) driven through a stub engine that answers with that reference; no GPU needed."""
import warnings

import numpy as np
import pytest
import torch
from scipy.optimize import minimize

from gpplus_b200._compat import NumericalWarning
from gpplus_b200.bayesian_optimizations import (optimize_acquisition_qbatch, optimize_knowledge_gradient,
                                                optimize_posterior_mean)
from gpplus_b200.models.gpregression import sobol_normal_samples
from kg_reference import kg_qbatch as reference_kg, kg_refit
from predict_grad_reference import predict_grad as reference_predict_grad
from problems import make_candidates, make_hyper, make_problem
from test_qacq import _AcqEngine
from test_qbatch_posterior import _batch, _model


class _KgEngine(_AcqEngine):
    """Adds kg_qbatch and predict_grad, answered by the references, with an optional forced jitter; records the
    arguments of kg_qbatch."""

    def predict_grad(self, xq, level_idx=None, noise_idx=None, mean_idx=None, include_noise=False, min_var=1e-10):
        self.calls.append("predict_grad")
        return reference_predict_grad(self.p, self.h, self._cand(xq, level_idx, noise_idx, mean_idx), include_noise,
                                      min_var)

    def kg_qbatch(self, xq, q, n_fantasies, base_samples, maximize=True, want_grad=True, level_idx=None,
                  noise_idx=None, mean_idx=None):
        self.calls.append("kg_qbatch")
        self.kg = dict(xq=xq, q=q, nf=n_fantasies, E=np.asarray(base_samples), maximize=maximize, want_grad=want_grad,
                       level_idx=level_idx, noise_idx=noise_idx, mean_idx=mean_idx)
        b = xq.shape[0] // (q + n_fantasies)
        jit = None if self.jitter is None else np.asarray(self.jitter)[:b]
        v, d, jit = reference_kg(self.p, self.h, self._cand(xq, level_idx, noise_idx, mean_idx), q, n_fantasies,
                                 base_samples, maximize, jit)
        return v, (d if want_grad else None), jit


def _case(kernel, mixed=False, seed=0):
    if mixed:
        p = make_problem(30, 2, kernel, dz=2, n_combo=3, n_noise=2, n_mean=2, seed=seed, n_pass=3)
    else:
        p = make_problem(30, 3, kernel, seed=seed)
    return p, make_hyper(p, noise=1e-2)


def _jitter_case():
    """t-batch 1's actual rows repeat one point far from the training set, in a noise group without noise, and its
    fantasy solutions lie near it: with sigma_f^2 = 1 its A is exactly the all-ones matrix, which needs the 1e-8 rung,
    while c_f is not zero."""
    p = make_problem(30, 3, 2, n_noise=2, seed=4)
    p["noise_idx"] = np.zeros(30, dtype=np.int32)
    h = make_hyper(p, noise=1e-2)
    h["sigma_f2"] = 1.0
    h["noise"] = np.array([1e-2, 0.0])
    q, nf = 3, 4
    c = make_candidates(p, 3 * (q + nf), seed=8)
    c["noise_idx"] = np.zeros(3 * (q + nf), dtype=np.int32)
    r = q + nf
    c["xq"][r:r + q] = 1e3
    c["xq"][r + q:2 * r] = 1e3 + 0.3 * np.random.default_rng(1).standard_normal((nf, 3))
    c["noise_idx"][r:r + q] = 1
    return p, h, c, q, nf


@pytest.mark.parametrize("maximize", [True, False])
@pytest.mark.parametrize("kernel,mixed", [(0, False), (1, False), (2, False), (1, True)])
def test_closed_form_equals_refit_semantics(kernel, mixed, maximize):
    p, h = _case(kernel, mixed)
    for q, nf in ((1, 1), (3, 4), (2, 6)):
        c = make_candidates(p, 3 * (q + nf), seed=3 + q)
        E = sobol_normal_samples(nf, q, seed=q).numpy()
        v, d, jit = reference_kg(p, h, c, q, nf, E, maximize)
        assert v.shape == (3,) and d.shape == (3 * (q + nf), p["dq"]) and (jit == 0).all()
        np.testing.assert_allclose(v, kg_refit(p, h, c, q, nf, E, maximize), rtol=0, atol=1e-10)


def test_closed_form_equals_refit_semantics_with_jitter():
    p, h, c, q, nf = _jitter_case()
    E = sobol_normal_samples(nf, q, seed=2).numpy()
    for maximize in (True, False):
        v, _, jit = reference_kg(p, h, c, q, nf, E, maximize)
        np.testing.assert_array_equal(jit, [0.0, 1e-8, 0.0])
        np.testing.assert_allclose(v, kg_refit(p, h, c, q, nf, E, maximize), rtol=0, atol=1e-10)


@pytest.mark.parametrize("mixed", [False, True])
def test_reference_gradient_matches_central_differences(mixed):
    p, h = _case(1, mixed, seed=2)
    q, nf = 2, 3
    c = make_candidates(p, 2 * (q + nf), seed=5)
    E = sobol_normal_samples(nf, q, seed=1).numpy()
    _, d, _ = reference_kg(p, h, c, q, nf, E)
    eps = 1e-6
    fd = np.zeros_like(d)
    for r in range(d.shape[0]):
        for k in range(p["dq"]):
            vals = []
            for s in (1.0, -1.0):
                cc = dict(c)
                cc["xq"] = np.array(c["xq"])
                cc["xq"][r, k] += s * eps
                vals.append(kg_refit(p, h, cc, q, nf, E).sum())
            fd[r, k] = (vals[0] - vals[1]) / (2 * eps)
    assert np.abs(d[:q]).max() > 1e-3 and np.abs(d[q:q + nf]).max() > 1e-3  # actual and fantasy rows both move
    np.testing.assert_allclose(d, fd, rtol=1e-5, atol=1e-8)


def _scaled(stub):
    a = stub.kg
    return reference_kg(stub.p, stub.h, stub._cand(a["xq"], a["level_idx"], a["noise_idx"], a["mean_idx"]), a["q"],
                        a["nf"], a["E"], a["maximize"])


@pytest.mark.parametrize("maximize", [True, False])
@pytest.mark.parametrize("kind", ["quant", "mixed"])
def test_values_current_value_cost_and_gradients_in_y_units(kind, maximize):
    m, X = _model(kind)
    q, nf = 2, 3
    Xb = _batch(X, (2, 3, q + nf)).requires_grad_(True)
    stub = _KgEngine(m)
    y_min, y_std = float(m.y_min), float(m.y_std)
    assert abs(y_std - 1.0) > 0.5 and abs(y_min) > 0.5
    sgn = 1.0 if maximize else -1.0
    with m.engine_override(stub):
        v = m.knowledge_gradient(Xb, nf, maximize=maximize)
        v.sum().backward()
        v_sc, d_sc, _ = _scaled(stub)
        assert stub.kg["want_grad"] and stub.kg["q"] == q and stub.kg["nf"] == nf
        assert stub.kg["maximize"] is maximize
        np.testing.assert_allclose(v.detach().numpy().reshape(-1), sgn * y_min + y_std * v_sc, rtol=1e-13)
        cols = m._quant_columns()
        g = Xb.grad.reshape(-1, X.shape[1])
        np.testing.assert_allclose(g[:, cols].numpy(), y_std * d_sc, rtol=1e-12, atol=1e-14)
        assert bool((g[:, [c for c in range(X.shape[1]) if c not in cols]] == 0).all())
        assert v.shape == (2, 3) and v.dtype == torch.float64

        cur = sgn * y_min + 0.3
        with torch.no_grad():
            v2 = m.knowledge_gradient(Xb, nf, maximize=maximize, current_value=cur)
        np.testing.assert_allclose(v2.numpy(), v.detach().numpy() - cur, rtol=1e-14, atol=1e-14)
        if kind == "mixed":
            cost = {0: 10.0, 1: 1.5}
            with torch.no_grad():
                v3 = m.knowledge_gradient(Xb, nf, maximize=maximize, current_value=cur, cost_by_source=cost)
                v4 = m.knowledge_gradient(Xb, nf, maximize=maximize, current_value=cur, cost_by_source=[10.0, 1.5])
            src = Xb.detach()[..., :q, -1]
            total = (10.0 * (src == 0) + 1.5 * (src == 1)).sum(-1)
            np.testing.assert_allclose(v3.numpy(), (v2 / total).numpy(), rtol=1e-14)
            assert torch.equal(v3, v4)


def test_levels_noise_and_means_are_gathered_for_all_rows():
    m, X = _model("mixed")
    q, nf = 2, 2
    Xb = _batch(X, (3, q + nf))
    stub = _KgEngine(m)
    with m.engine_override(stub):
        m.knowledge_gradient(Xb, nf)
    rows = Xb.reshape(-1, X.shape[1]).double()
    a = stub.kg
    np.testing.assert_array_equal(a["level_idx"], m._level_index(rows, False))
    np.testing.assert_array_equal(a["noise_idx"], m._noise_index(rows))
    np.testing.assert_array_equal(a["mean_idx"], m._mean_index(rows))
    np.testing.assert_array_equal(a["xq"], rows[:, m._quant_columns()].numpy())
    assert a["want_grad"] is False


def test_default_base_samples_and_argument_errors():
    m, X = _model("quant")
    q, nf = 3, 5
    Xb = _batch(X, (2, q + nf))
    stub = _KgEngine(m)
    with m.engine_override(stub):
        v = m.knowledge_gradient(Xb, nf, seed=4)
        np.testing.assert_array_equal(stub.kg["E"], sobol_normal_samples(nf, q, 4).numpy())
        E = torch.randn(nf, q, dtype=torch.float64, generator=torch.Generator().manual_seed(0))
        m.knowledge_gradient(Xb, nf, base_samples=E)
        np.testing.assert_array_equal(stub.kg["E"], E.numpy())
        assert not torch.equal(v, m.knowledge_gradient(Xb, nf, base_samples=E))
        n_calls = stub.calls.count("kg_qbatch")
        for args, kw, match in (((nf,), dict(base_samples=E[:, :2]), "base_samples must have shape"),
                                ((q + nf,), {}, "q >= 1"),
                                ((0,), {}, "q >= 1"),
                                ((nf,), dict(cost_by_source={0: 1.0}), "cost_by_source needs current_value")):
            with pytest.raises(ValueError, match=match):
                m.knowledge_gradient(Xb, *args, **kw)
        with pytest.raises(ValueError, match="exceeds"):
            m.knowledge_gradient(_batch(X, (1, 129)), 64)
        with pytest.raises(ValueError, match="expects X"):
            m.knowledge_gradient(Xb[0, 0], 1)
        with pytest.raises(ValueError, match="kind must be one of"):
            m.acquisition_qbatch(_batch(X, (2, 2)), "qKG")
        assert stub.calls.count("kg_qbatch") == n_calls


def test_backward_scales_by_the_upstream_gradient_and_second_derivative_raises():
    m, X = _model("quant")
    q, nf = 2, 2
    Xb = _batch(X, (3, q + nf)).requires_grad_(True)
    stub = _KgEngine(m)
    w = torch.tensor([0.5, -2.0, 3.0], dtype=torch.float64)
    with m.engine_override(stub):
        v = m.knowledge_gradient(Xb, nf)
        g, = torch.autograd.grad((w * v).sum(), Xb)
        _, d_sc, _ = _scaled(stub)
        want = float(m.y_std) * w.reshape(3, 1, 1) * torch.as_tensor(d_sc).reshape(3, q + nf, -1)
        np.testing.assert_allclose(g.numpy(), want.numpy(), rtol=1e-12, atol=1e-14)
        v = m.knowledge_gradient(Xb, nf)
        g, = torch.autograd.grad(v.sum(), Xb, create_graph=True)
        with pytest.raises(RuntimeError):
            torch.autograd.grad(g.sum(), Xb)


def test_jitter_raises_a_numerical_warning():
    m, X = _model("quant")
    stub = _KgEngine(m)
    stub.jitter = np.array([0.0, 1e-7])
    with m.engine_override(stub), warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        m.knowledge_gradient(_batch(X, (2, 3)), 1)
    assert any(issubclass(x.category, NumericalWarning) for x in w)


def test_optimizer_returns_actual_rows_and_projects_the_fantasies():
    m, X = _model("mixed")
    stub = _KgEngine(m)
    seen = []
    orig = m.knowledge_gradient

    def spy(Xc, nf, **kw):
        assert nf == 3 and set(kw) == {"base_samples", "current_value", "cost_by_source"}
        seen.append(Xc.detach().clone())
        return orig(Xc, nf, **kw)

    m.knowledge_gradient = spy
    bounds = np.array([[-1.0, -0.5, 0.0], [1.0, 0.5, 2.0]])
    fixed = {3: 1.0, 4: 1.0}
    args = dict(fixed_columns=fixed, fantasy_fixed_columns={4: 0.0}, num_restarts=2, raw_samples=8,
                options={"maxiter": 4}, seed=1, current_value=0.0, cost_by_source={0: 5.0, 1: 1.0})
    with m.engine_override(stub):
        X1, v1 = optimize_knowledge_gradient(m, bounds, 2, num_fantasies=3, **args)
        n = len(seen)
        X2, v2 = optimize_knowledge_gradient(m, bounds, 2, num_fantasies=3, **args)
        with pytest.raises(ValueError, match="cannot be fixed"):
            optimize_knowledge_gradient(m, bounds, 2, num_fantasies=3, fixed_columns=fixed,
                                        fantasy_fixed_columns={0: 0.0})
    assert X1.shape == (2, 5) and np.isfinite(v1)
    assert torch.equal(X1, X2) and v1 == v2 and len(seen) == 2 * n
    for Xc in seen:
        assert Xc.shape[-2] == 5
        qv = Xc[..., :3]
        assert bool((qv >= torch.tensor(bounds[0])).all()) and bool((qv <= torch.tensor(bounds[1])).all())
        assert bool((Xc[..., 3] == 1.0).all())
        assert bool((Xc[..., :2, 4] == 1.0).all()) and bool((Xc[..., 2:, 4] == 0.0).all())
    assert bool((X1[:, 3] == 1.0).all()) and bool((X1[:, 4] == 1.0).all())
    with m.engine_override(stub), torch.no_grad():  # the value is that of a batch whose actual rows are returned
        assert any(torch.equal(Xc[i, :2], X1) for Xc in seen for i in range(Xc.shape[0]))


def test_optimize_posterior_mean_through_predict():
    m, X = _model("mixed")
    stub = _KgEngine(m)
    bounds = np.array([[-1.0, -0.5, 0.0], [1.0, 0.5, 2.0]])
    with m.engine_override(stub):
        for maximize in (True, False):
            x, v = optimize_posterior_mean(m, bounds, fixed_columns={3: 0.0, 4: 0.0}, maximize=maximize,
                                           num_restarts=2, raw_samples=16, options={"maxiter": 10}, seed=3)
            assert x.shape == (5,) and x[3] == 0.0 and x[4] == 0.0
            with torch.no_grad():
                mu = float(m.predict(x[None], return_std=False)[0])
            assert v == pytest.approx((1.0 if maximize else -1.0) * mu, rel=1e-14, abs=1e-14)


def _optimize_acquisition_qbatch_before(model, bounds, q, kind, fixed_columns=None, num_restarts=8, raw_samples=256,
                                        options=None, seed=0, **acq_kwargs):
    """optimize_acquisition_qbatch as it was before its screening and L-BFGS-B run moved into a shared helper."""
    q = int(q)
    d = int(model.train_inputs[0].shape[1])
    cols = list(model._quant_columns())
    fixed = dict(fixed_columns or {})
    lo, hi = (torch.as_tensor(np.asarray(bounds, dtype=np.float64)).reshape(2, -1)[k] for k in (0, 1))
    dq = len(cols)
    acq_kwargs = dict(acq_kwargs)
    if kind != "qNIPV" and acq_kwargs.get("base_samples") is None:
        n_b = 0
        if acq_kwargs.get("X_baseline") is not None:
            n_b = int(torch.as_tensor(acq_kwargs["X_baseline"]).reshape(-1, d).shape[0])
        acq_kwargs["base_samples"] = sobol_normal_samples(acq_kwargs.pop("num_samples", 512), q + n_b, seed)
    acq_kwargs.pop("num_samples", None)

    def full(z):
        X = torch.zeros(z.shape[0], q, d, dtype=torch.float64)
        X[:, :, cols] = z
        for c, v in fixed.items():
            X[:, :, c] = float(v)
        return X

    raw = torch.quasirandom.SobolEngine(dimension=q * dq, scramble=True, seed=int(seed)).draw(int(raw_samples),
                                                                                          dtype=torch.float64)
    z_raw = lo + (hi - lo) * raw.reshape(-1, q, dq)
    with torch.no_grad():
        v_raw = model.acquisition_qbatch(full(z_raw), kind, **acq_kwargs).double().numpy()
    k = min(int(num_restarts), z_raw.shape[0])
    order = np.lexsort((np.arange(len(v_raw)), -v_raw))[:k]
    z0 = z_raw[torch.as_tensor(order)].numpy()

    def neg(flat):
        z = torch.tensor(flat.reshape(k, q, dq), dtype=torch.float64)
        X = full(z).requires_grad_(True)
        v = model.acquisition_qbatch(X, kind, **acq_kwargs).sum()
        g, = torch.autograd.grad(v, X)
        return -float(v.detach()), -g[:, :, cols].numpy().reshape(-1).astype(np.float64)

    box = list(zip(np.tile(lo.numpy(), k * q), np.tile(hi.numpy(), k * q)))
    res = minimize(neg, z0.reshape(-1), jac=True, method="L-BFGS-B", bounds=box, options=options)
    z_opt = torch.tensor(np.clip(res.x.reshape(k, q, dq), lo.numpy(), hi.numpy()), dtype=torch.float64)
    with torch.no_grad():
        v_opt = model.acquisition_qbatch(full(z_opt), kind, **acq_kwargs).double().numpy()
    best = int(np.lexsort((np.arange(k), -v_opt))[0])
    return full(z_opt[best:best + 1])[0], float(v_opt[best])


@pytest.mark.parametrize("kind,kw", [("qEI", dict(best_f=5.0)), ("qUCB", dict(beta=0.7))])
def test_optimize_acquisition_qbatch_is_unchanged(kind, kw):
    m, X = _model("mixed")
    bounds = np.array([[-1.0, -0.5, 0.0], [1.0, 0.5, 2.0]])
    args = dict(fixed_columns={3: 2.0, 4: 0.0}, num_restarts=3, raw_samples=16, options={"maxiter": 6}, seed=2,
                num_samples=32, **kw)
    with m.engine_override(_KgEngine(m)):
        X1, v1 = optimize_acquisition_qbatch(m, bounds, 2, kind, **args)
        X0, v0 = _optimize_acquisition_qbatch_before(m, bounds, 2, kind, **args)
    assert torch.equal(X1, X0) and v1 == v0
