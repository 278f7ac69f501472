"""Batch integrated posterior variance (qNIPV): the CPU reference against botorch's refit semantics and central
differences, and the host side (GPR.acquisition_qbatch(X, "qNIPV", mc_points), the autograd Function behind it and
optimize_acquisition_qbatch) driven through a stub engine that answers with that reference; no GPU needed."""
import warnings

import numpy as np
import pytest
import torch

from gpplus_b200._compat import NumericalWarning
from gpplus_b200.bayesian_optimizations import optimize_acquisition_qbatch
from nipv_reference import nipv_qbatch as reference_nipv, nipv_refit
from problems import make_candidates, make_hyper, make_problem
from test_qbatch_posterior import _QBatchEngine, _batch, _model


class _NipvEngine(_QBatchEngine):
    """Adds ipv_points / nipv_qbatch, answered by the reference, and records their arguments."""

    def ipv_points(self, xq, level_idx=None):
        self.calls.append("ipv_points")
        self.ipv = {"m": xq.shape[0], "xq": np.array(xq), "level_idx": None if level_idx is None else
                    np.array(level_idx)}

    def nipv_qbatch(self, xq, q, want_grad=True, level_idx=None, noise_idx=None):
        self.calls.append("nipv_qbatch")
        self.nipv = dict(xq=xq, q=q, want_grad=want_grad, level_idx=level_idx, noise_idx=noise_idx)
        v, d, jit = reference_nipv(self.p, self.h, self._cand(xq, level_idx, noise_idx, None), self.ipv, q)
        return v, (d if want_grad else None), jit


def _case(kernel, latent=False, seed=0):
    if latent:
        p = make_problem(30, 2, kernel, dz=2, n_combo=3, n_noise=2, n_mean=1, seed=seed, n_pass=3)
    else:
        p = make_problem(30, 3, kernel, seed=seed)
    h = make_hyper(p, noise=1e-2)
    return p, h


@pytest.mark.parametrize("kernel,latent", [(0, False), (1, False), (2, False), (2, True)])
def test_closed_form_equals_refit_semantics(kernel, latent):
    p, h = _case(kernel, latent)
    q = 3
    cand = make_candidates(p, 4 * q, seed=3)
    ipv = make_candidates(p, 17, seed=4)
    v, d, jit = reference_nipv(p, h, cand, ipv, q)
    assert v.shape == (4,) and d.shape == (4 * q, p["dq"]) and (jit == 0).all()
    np.testing.assert_allclose(v, nipv_refit(p, h, cand, ipv, q), rtol=0, atol=1e-10)
    assert (v < 0).all()


@pytest.mark.parametrize("latent", [False, True])
def test_reference_gradient_matches_central_differences(latent):
    p, h = _case(1, latent, seed=2)
    q = 2
    cand = make_candidates(p, 2 * q, seed=5)
    ipv = make_candidates(p, 9, seed=6)
    _, d, _ = reference_nipv(p, h, cand, ipv, q)
    eps = 1e-6
    fd = np.zeros_like(d)
    for r in range(2 * q):
        for c in range(p["dq"]):
            vals = []
            for s in (1.0, -1.0):
                cc = dict(cand)
                cc["xq"] = np.array(cand["xq"])
                cc["xq"][r, c] += s * eps
                vals.append(nipv_refit(p, h, cc, ipv, q).sum())
            fd[r, c] = (vals[0] - vals[1]) / (2 * eps)
    np.testing.assert_allclose(d, fd, rtol=1e-5, atol=1e-8)


def _points(X, M, seed=9):
    return _batch(X, (M,), seed=seed)


@pytest.mark.parametrize("kind", ["quant", "mixed"])
def test_values_and_gradients_in_y_units(kind):
    m, X = _model(kind)
    Xb = _batch(X, (3, 2)).requires_grad_(True)
    P = _points(X, 11)
    stub = _NipvEngine(m)
    with m.engine_override(stub):
        v = m.acquisition_qbatch(Xb, "qNIPV", mc_points=P)
        v.sum().backward()
    assert v.shape == (3,) and v.dtype == torch.float64
    a = stub.nipv
    assert a["want_grad"] and a["q"] == 2
    v_sc, d_sc, _ = reference_nipv(stub.p, stub.h, stub._cand(a["xq"], a["level_idx"], a["noise_idx"], None),
                                   stub.ipv, 2)
    s2 = float(m.y_std) ** 2
    assert abs(s2 - 1.0) > 1.0
    np.testing.assert_allclose(v.detach().numpy(), s2 * v_sc, rtol=1e-13)
    cols = m._quant_columns()
    g = Xb.grad.reshape(-1, X.shape[1])
    np.testing.assert_allclose(g[:, cols].numpy(), s2 * d_sc, rtol=1e-12, atol=1e-14)
    other = [c for c in range(X.shape[1]) if c not in cols]
    assert bool((g[:, other] == 0).all())
    if kind == "mixed":  # the candidates are fantasised with their own source's noise group
        np.testing.assert_array_equal(a["noise_idx"], m._noise_index(Xb.detach().reshape(-1, X.shape[1])))


def test_argument_checks_per_kind():
    m, X = _model("quant")
    Xb = _batch(X, (2, 2))
    P = _points(X, 5)
    stub = _NipvEngine(m)
    with m.engine_override(stub):
        with pytest.raises(ValueError, match="needs mc_points"):
            m.acquisition_qbatch(Xb, "qNIPV")
        for kw in (dict(best_f=1.0), dict(beta=0.5), dict(X_baseline=P[:2]), dict(base_samples=torch.zeros(4, 2))):
            with pytest.raises(ValueError, match="qNIPV takes no"):
                m.acquisition_qbatch(Xb, "qNIPV", mc_points=P, **kw)
        for kind, kw in (("qEI", dict(best_f=1.0)), ("qUCB", dict(beta=1.0)), ("qNEI", dict(X_baseline=P[:2]))):
            with pytest.raises(ValueError, match="mc_points is for qNIPV only"):
                m.acquisition_qbatch(Xb, kind, mc_points=P, **kw)
        with pytest.raises(ValueError, match="mc_points must have shape"):
            m.acquisition_qbatch(Xb, "qNIPV", mc_points=P[:, :2])
        with pytest.raises(ValueError, match="kind must be one of"):
            m.acquisition_qbatch(Xb, "qKG", mc_points=None)
    assert "nipv_qbatch" not in stub.calls and "ipv_points" not in stub.calls


def test_mc_points_levels_are_ranked_with_the_candidates():
    m, X = _model("mixed")
    Xb = _batch(X, (2, 3))
    P = _points(X, 7)
    P[:, 4] = 1.0  # integrate the variance of one source
    stub = _NipvEngine(m)
    with m.engine_override(stub):
        m.acquisition_qbatch(Xb, "qNIPV", mc_points=P)
    rows = torch.cat([Xb.reshape(-1, X.shape[1]), P]).double()
    want = m._level_index(rows, False)
    np.testing.assert_array_equal(stub.nipv["level_idx"], want[:6])
    np.testing.assert_array_equal(stub.ipv["level_idx"], want[6:])
    np.testing.assert_array_equal(stub.ipv["xq"], rows[6:, m._quant_columns()].numpy())


def test_integration_set_is_stored_once_per_factor_points_and_engine():
    m, X = _model("quant")
    P = _points(X, 6)
    stub = _NipvEngine(m)
    with m.engine_override(stub):
        for s in range(3):
            x = _batch(X, (2, 2), seed=s).requires_grad_(s == 1)
            m.acquisition_qbatch(x, "qNIPV", mc_points=P).sum()
        assert stub.calls.count("ipv_points") == 1 and stub.calls.count("nipv_qbatch") == 3
        m.acquisition_qbatch(_batch(X, (2, 2)), "qNIPV", mc_points=P + 0.1)  # new points
        assert stub.calls.count("ipv_points") == 2
        with torch.no_grad():  # a refit: new hyper-parameters, a new factor
            m.covar_module.raw_outputscale.add_(0.3)
        m.acquisition_qbatch(_batch(X, (2, 2)), "qNIPV", mc_points=P + 0.1)
        assert stub.calls.count("ipv_points") == 3 and stub.calls.count("factorize") == 2
        m.acquisition_qbatch(_batch(X, (2, 2)), "qNIPV", mc_points=P + 0.1)
        assert stub.calls.count("ipv_points") == 3
    other = _NipvEngine(m)
    with m.engine_override(other):  # a new handle holds no set
        m.acquisition_qbatch(_batch(X, (2, 2)), "qNIPV", mc_points=P + 0.1)
    assert other.calls.count("ipv_points") == 1


def test_jitter_raises_a_numerical_warning():
    m, X = _model("quant")

    class _Jit(_NipvEngine):
        def nipv_qbatch(self, *a, **k):
            v, d, jit = super().nipv_qbatch(*a, **k)
            return v, d, np.where(np.arange(len(jit)) == 1, 1e-7, 0.0)

    stub = _Jit(m)
    with m.engine_override(stub), warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        m.acquisition_qbatch(_batch(X, (2, 2)), "qNIPV", mc_points=_points(X, 4))
    assert any(issubclass(x.category, NumericalWarning) for x in w)


def test_optimizer_draws_no_base_samples_and_keeps_bounds_and_fixed_columns():
    m, X = _model("mixed")
    stub = _NipvEngine(m)
    seen = []
    orig = m.acquisition_qbatch

    def spy(Xc, kind, **kw):
        assert kind == "qNIPV" and set(kw) == {"mc_points"}
        seen.append(Xc.detach().clone())
        return orig(Xc, kind, **kw)

    m.acquisition_qbatch = spy
    bounds = np.array([[-1.0, -0.5, 0.0], [1.0, 0.5, 2.0]])
    fixed = {3: 1.0, 4: 0.0}
    P = _points(X, 8)
    with m.engine_override(stub):
        X1, v1 = optimize_acquisition_qbatch(m, bounds, 2, "qNIPV", fixed_columns=fixed, num_restarts=2,
                                             raw_samples=8, options={"maxiter": 4}, seed=1, mc_points=P)
    assert X1.shape == (2, 5) and np.isfinite(v1)
    for Xc in seen + [X1[None]]:
        q = Xc[..., :3]
        assert bool((q >= torch.tensor(bounds[0])).all()) and bool((q <= torch.tensor(bounds[1])).all())
        assert bool((Xc[..., 3] == 1.0).all()) and bool((Xc[..., 4] == 0.0).all())
    assert stub.calls.count("ipv_points") == 1
