"""Host side of the joint posterior (GPR.predict_joint / GPR.sample_posterior and their GP_Plus overrides), driven
through a stub engine that answers with the CPU reference (no GPU needed), and the pin of that reference."""
import warnings

import numpy as np
import pytest
import torch

from gpplus_b200._compat import NumericalWarning
from gpplus_b200.models import GP_Plus
from joint_posterior_reference import joint_factor, predict_joint as reference_predict_joint
from oracle import gp_oracle as O
from problems import make_candidates, make_hyper, make_problem


class _JointEngine:
    """Answers factorize / predict / predict_joint / sample_posterior of the model's training set with the CPU
    references; ``jitter`` is what sample_posterior reports."""

    def __init__(self, model, jitter=0.0):
        kw = model._engine_kwargs(0)
        xq = kw["xq"] if kw["xq"] is not None else np.zeros((len(kw["y"]), 0))
        self.dq, self.dz, self.n_mean, self.n_pass = xq.shape[1], kw["dz"], kw["n_mean"], kw["n_pass"]
        self.p = {"n": len(kw["y"]), "dq": self.dq, "dz": self.dz, "n_combo": kw["n_combo"], "n_noise": kw["n_noise"],
                  "n_mean": self.n_mean, "kernel": kw["kernel"], "xq": xq, "y": kw["y"], "level_idx": kw["level_idx"],
                  "noise_idx": kw["noise_idx"], "mean_idx": kw["mean_idx"], "n_pass": self.n_pass}
        self.jitter = jitter
        self.calls = []

    def factorize(self, hyper):
        self.h = hyper

    def _cand(self, xq, level_idx, noise_idx, mean_idx):
        return {"m": xq.shape[0], "xq": xq, "level_idx": level_idx, "noise_idx": noise_idx, "mean_idx": mean_idx}

    def predict(self, xq, level_idx=None, noise_idx=None, mean_idx=None, include_noise=False, min_var=1e-10):
        self.calls.append(("predict", include_noise))
        return O.predict(self.p, self.h, self._cand(xq, level_idx, noise_idx, mean_idx), include_noise, min_var)

    def predict_joint(self, xq, level_idx=None, noise_idx=None, mean_idx=None, include_noise=False):
        self.calls.append(("predict_joint", include_noise))
        return reference_predict_joint(self.p, self.h, self._cand(xq, level_idx, noise_idx, mean_idx), include_noise)

    def sample_posterior(self, xq, base_samples, level_idx=None, noise_idx=None, mean_idx=None, include_noise=False):
        self.calls.append(("sample_posterior", include_noise))
        self.base = np.array(base_samples, copy=True)
        mu, cov = reference_predict_joint(self.p, self.h, self._cand(xq, level_idx, noise_idx, mean_idx),
                                          include_noise)
        L = np.linalg.cholesky(cov + self.jitter * np.eye(len(mu)))
        return mu[None, :] + base_samples @ L.T, self.jitter


def _model(kind):
    rng = np.random.default_rng(3)
    n = 40
    X = np.hstack([rng.standard_normal((n, 3)), rng.integers(0, 3, (n, 1)), rng.integers(0, 2, (n, 1))]).astype(float)
    y = 5.0 + 3.0 * np.sin(X[:, 0]) + 0.3 * X[:, 3] + 0.2 * X[:, 4] + 0.05 * rng.standard_normal(n)
    if kind == "quant":
        m = GP_Plus(torch.tensor(X[:, :3]), torch.tensor(y), dtype=torch.float64,
                    quant_correlation_class="Matern52Kernel")
    else:
        m = GP_Plus(torch.tensor(X), torch.tensor(y), qual_dict={3: 3, 4: 2}, multiple_noise=True,
                    m_gp="multiple_constant", dtype=torch.float64)
    Xq = X[:7, : m.train_inputs[0].shape[1]].copy()
    Xq[:, :3] += 0.3 * rng.standard_normal((7, 3))
    return m, torch.tensor(Xq)


def _engine_cand(m, Xq, include_noise):
    cols = m._quant_columns()
    return {"m": Xq.shape[0], "xq": Xq[:, cols].numpy(), "level_idx": m._level_index(Xq, False),
            "noise_idx": m._noise_index(Xq) if include_noise else None, "mean_idx": m._mean_index(Xq)}


@pytest.mark.parametrize("kind", ["quant", "mixed"])
@pytest.mark.parametrize("include_noise", [False, True])
def test_joint_outputs_are_in_original_y_units(kind, include_noise):
    m, Xq = _model(kind)
    stub = _JointEngine(m)
    with m.engine_override(stub):
        mean, cov = m.predict_joint(Xq, include_noise=include_noise)
        E = torch.randn(5, Xq.shape[0], generator=torch.Generator().manual_seed(1), dtype=torch.float64)
        draws = m.sample_posterior(Xq, num_samples=5, include_noise=include_noise, base_samples=E)
        mean0, std0 = m.predict(Xq, return_std=True, include_noise=include_noise)
    assert not mean.requires_grad and not cov.requires_grad and not draws.requires_grad
    mu_sc, cov_sc = reference_predict_joint(stub.p, stub.h, _engine_cand(m, Xq, include_noise), include_noise)
    y_min, y_std = float(m.y_min), float(m.y_std)
    assert abs(y_std - 1.0) > 1.0 and abs(y_min) > 0.5  # the scaling is visible
    np.testing.assert_allclose(mean.numpy(), y_min + y_std * mu_sc, rtol=1e-14, atol=0)
    np.testing.assert_allclose(cov.numpy(), y_std ** 2 * cov_sc, rtol=1e-14, atol=0)
    assert torch.equal(mean, mean0)
    np.testing.assert_allclose(cov.diagonal().sqrt().numpy(), std0.numpy(), rtol=1e-10)
    L = np.linalg.cholesky(cov_sc)
    np.testing.assert_allclose(draws.numpy(), y_min + y_std * (mu_sc[None, :] + E.numpy() @ L.T), rtol=1e-13)


def test_default_base_samples_follow_the_generator():
    m, Xq = _model("mixed")
    stub = _JointEngine(m)
    with m.engine_override(stub):
        a = m.sample_posterior(Xq, num_samples=4, generator=torch.Generator().manual_seed(7))
        base_a = stub.base
        b = m.sample_posterior(Xq, num_samples=4, generator=torch.Generator().manual_seed(7))
        c = m.sample_posterior(Xq, num_samples=4, generator=torch.Generator().manual_seed(8))
    assert a.shape == (4, Xq.shape[0]) and a.dtype == torch.float64
    assert torch.equal(a, b) and not torch.equal(a, c)
    # gpytorch's rsample: randn(sample_shape + event_shape) in the covariance's dtype on its device
    expect = torch.randn(4, Xq.shape[0], generator=torch.Generator().manual_seed(7), dtype=torch.float64)
    assert np.array_equal(base_a, expect.numpy())


@pytest.mark.parametrize("shape", [(3,), (2, 7), (3, 6), (3, 7, 1)])
def test_wrong_base_sample_shape_raises(shape):
    m, Xq = _model("quant")
    stub = _JointEngine(m)
    with m.engine_override(stub):
        with pytest.raises(ValueError, match="base_samples"):
            m.sample_posterior(Xq, num_samples=3, base_samples=torch.zeros(shape, dtype=torch.float64))
    assert not any(c[0] == "sample_posterior" for c in stub.calls)


def test_jitter_warns_like_psd_safe_cholesky():
    m, Xq = _model("quant")
    with m.engine_override(_JointEngine(m, jitter=1e-7)):
        with pytest.warns(NumericalWarning, match="added jitter of 1.0e-07"):
            m.sample_posterior(Xq, num_samples=2)
    with m.engine_override(_JointEngine(m, jitter=0.0)):
        with warnings.catch_warnings():
            warnings.simplefilter("error", NumericalWarning)
            m.sample_posterior(Xq, num_samples=2)


def test_gp_plus_defaults():
    m, Xq = _model("mixed")
    stub = _JointEngine(m)
    with m.engine_override(stub):
        mean, cov = m.predict_joint(Xq.float())  # data_type_check casts to float64
        draws = m.sample_posterior(Xq)
    assert [c for c in stub.calls] == [("predict_joint", False), ("sample_posterior", False)]
    assert mean.dtype == torch.float64 and cov.shape == (Xq.shape[0], Xq.shape[0])
    assert draws.shape == (1, Xq.shape[0])


def test_predict_and_posterior_never_call_the_joint_entries():
    m, Xq = _model("mixed")
    stub = _JointEngine(m)
    with m.engine_override(stub):
        m.predict(Xq, return_std=True, include_noise=True)
        m.posterior(Xq)
    assert all(c[0] == "predict" for c in stub.calls) and len(stub.calls) == 2


@pytest.mark.parametrize("include_noise", [False, True])
def test_reference_diagonal_is_the_unclamped_oracle_variance(include_noise):
    p = make_problem(60, 3, 2, dz=2, n_combo=4, n_noise=2, n_mean=2, seed=4)
    h = make_hyper(p, seed=2, noise=1e-2)
    c = make_candidates(p, 25, seed=3)
    c["xq"][:3] = p["xq"][:3]  # some candidates on training points: variances near the noise level
    mu, cov = reference_predict_joint(p, h, c, include_noise)
    mu0, var0 = O.predict(p, h, c, include_noise, min_var=-np.inf)
    assert np.array_equal(mu, mu0)
    np.testing.assert_allclose(np.diag(cov), var0, rtol=0, atol=1e-15)
    assert np.array_equal(cov, cov.T)
    L, jit = joint_factor(cov)
    assert jit == 0.0
    np.testing.assert_allclose(L @ L.T, cov, atol=1e-14)
