"""Host side of the t-batch joint posterior (GPR.posterior on [..., q, d] inputs, the autograd Function behind it and
MultivariateNormal.rsample), driven through a stub engine that answers with the CPU reference (no GPU needed), and the
pin of that reference."""
import warnings

import numpy as np
import pytest
import torch

from gpplus_b200._compat import MultivariateNormal, NumericalWarning
from gpplus_b200.models import GP_Plus
from joint_posterior_reference import predict_joint as reference_predict_joint
from oracle import gp_oracle as O
from problems import make_candidates, make_hyper, make_problem
from qbatch_posterior_reference import posterior_qbatch as reference_posterior_qbatch


class _QBatchEngine:
    """Answers factorize / predict / posterior_qbatch / posterior_qbatch_grad of the model's training set with the CPU
    references and records the calls."""

    def __init__(self, model):
        kw = model._engine_kwargs(0)
        xq = kw["xq"] if kw["xq"] is not None else np.zeros((len(kw["y"]), 0))
        self.dq, self.dz, self.n_mean, self.n_pass = xq.shape[1], kw["dz"], kw["n_mean"], kw["n_pass"]
        self.p = {"n": len(kw["y"]), "dq": self.dq, "dz": self.dz, "n_combo": kw["n_combo"], "n_noise": kw["n_noise"],
                  "n_mean": self.n_mean, "kernel": kw["kernel"], "xq": xq, "y": kw["y"], "level_idx": kw["level_idx"],
                  "noise_idx": kw["noise_idx"], "mean_idx": kw["mean_idx"], "n_pass": self.n_pass}
        self.calls = []

    def factorize(self, hyper):
        self.calls.append("factorize")
        self.h = hyper

    def _cand(self, xq, level_idx, noise_idx, mean_idx):
        return {"m": xq.shape[0], "xq": xq, "level_idx": level_idx, "noise_idx": noise_idx, "mean_idx": mean_idx}

    def predict(self, xq, level_idx=None, noise_idx=None, mean_idx=None, include_noise=False, min_var=1e-10):
        self.calls.append("predict")
        return O.predict(self.p, self.h, self._cand(xq, level_idx, noise_idx, mean_idx), include_noise, min_var)

    def posterior_qbatch(self, xq, q, level_idx=None, noise_idx=None, mean_idx=None, include_noise=False):
        self.calls.append("posterior_qbatch")
        self.last = self._cand(xq, level_idx, noise_idx, mean_idx)
        mean, cov, _ = reference_posterior_qbatch(self.p, self.h, self.last, q, include_noise)
        return mean, cov

    def posterior_qbatch_grad(self, xq, q, g_mean, g_cov, level_idx=None, noise_idx=None, mean_idx=None,
                              include_noise=False):
        self.calls.append("posterior_qbatch_grad")
        self.g = (g_mean, g_cov)
        _, _, d = reference_posterior_qbatch(self.p, self.h, self._cand(xq, level_idx, noise_idx, mean_idx), q,
                                             include_noise, g_mean, g_cov)
        return d


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
    return m, X[:, : m.train_inputs[0].shape[1]]


def _batch(X, shape, seed=5):
    """Candidates of shape [*shape, d]: training rows with perturbed quantitative inputs."""
    rng = np.random.default_rng(seed)
    rows = rng.integers(0, X.shape[0], int(np.prod(shape)))
    Xq = X[rows].copy()
    Xq[:, :3] += 0.3 * rng.standard_normal((len(rows), 3))
    return torch.tensor(Xq.reshape(*shape, X.shape[1]))


@pytest.mark.parametrize("kind", ["quant", "mixed"])
@pytest.mark.parametrize("shape", [(1, 4), (5, 3), (2, 3, 2)])
@pytest.mark.parametrize("observation_noise", [False, True])
def test_shapes_and_scaled_units(kind, shape, observation_noise):
    m, X = _model(kind)
    Xb = _batch(X, shape)
    q = shape[-1]
    stub = _QBatchEngine(m)
    with m.engine_override(stub):
        post = m.posterior(Xb, observation_noise=observation_noise)
        mean0, std0 = m.predict(Xb.reshape(-1, Xb.shape[-1]), return_std=True, include_noise=observation_noise)
    assert post.mean.shape == Xb.shape[:-1] and post.covariance_matrix.shape == Xb.shape[:-1] + (q,)
    assert post.mean.dtype == torch.float64 and not post.mean.requires_grad
    assert stub.calls.count("posterior_qbatch") == 1
    y_min, y_std = float(m.y_min), float(m.y_std)
    assert abs(y_std - 1.0) > 1.0 and abs(y_min) > 0.5  # the scaling would be visible
    flat_mean = post.mean.reshape(-1).numpy()
    np.testing.assert_allclose(y_min + y_std * flat_mean, mean0.numpy(), rtol=1e-13)
    var = torch.diagonal(post.covariance_matrix, dim1=-2, dim2=-1).reshape(-1)
    np.testing.assert_allclose((var.sqrt() * y_std).numpy(), std0.numpy(), rtol=1e-10)
    # every block is the joint posterior of its own q rows (the gather of levels, groups and means is predict's)
    c = stub.last
    covs = post.covariance_matrix.reshape(-1, q, q).numpy()
    for t in range(covs.shape[0]):
        sub = {k: (v[t * q:(t + 1) * q] if isinstance(v, np.ndarray) else v) for k, v in c.items()}
        sub["m"] = q
        _, ref = reference_predict_joint(stub.p, stub.h, sub, observation_noise)
        np.testing.assert_allclose(covs[t], ref, rtol=0, atol=1e-14)


def test_two_dimensional_inputs_keep_the_marginal_path():
    m, X = _model("mixed")
    Xq = _batch(X, (6,))
    stub = _QBatchEngine(m)
    with m.engine_override(stub):
        post = m.posterior(Xq)
        m.predict(Xq, return_std=True, include_noise=True)
    assert [c for c in stub.calls if c != "factorize"] == ["predict", "predict"]
    assert post.mean.shape == (6,) and post.covariance_matrix.shape == (6, 6)
    cov = post.covariance_matrix
    assert torch.equal(cov, torch.diag(torch.diagonal(cov)))


def test_categorical_columns_are_ranked_against_all_rows():
    m, X = _model("mixed")
    Xb = _batch(X, (3, 4))
    stub = _QBatchEngine(m)
    with m.engine_override(stub):
        m.posterior(Xb)
    flat = Xb.reshape(-1, Xb.shape[-1])
    assert np.array_equal(stub.last["level_idx"], m._level_index(flat, False))
    assert np.array_equal(stub.last["mean_idx"], m._mean_index(flat))


@pytest.mark.parametrize("kind", ["quant", "mixed"])
def test_gradient_maps_to_quantitative_columns(kind):
    m, X = _model(kind)
    Xb = _batch(X, (2, 3, 2), seed=8).requires_grad_(True)
    stub = _QBatchEngine(m)
    rng = np.random.default_rng(2)
    a = torch.tensor(rng.standard_normal((2, 3, 2)))
    G = torch.tensor(rng.standard_normal((2, 3, 2, 2)))
    with m.engine_override(stub):
        post = m.posterior(Xb, observation_noise=False)
        loss = (a * post.mean).sum() + (G * post.covariance_matrix).sum()
        loss.backward()
    assert stub.calls[-1] == "posterior_qbatch_grad"
    g_mean, g_cov = stub.g
    np.testing.assert_array_equal(np.asarray(g_mean).reshape(-1), a.numpy().reshape(-1))
    np.testing.assert_array_equal(np.asarray(g_cov).reshape(-1), G.numpy().reshape(-1))
    cols = m._quant_columns()
    flat = Xb.detach().reshape(-1, Xb.shape[-1])
    cand = {"m": flat.shape[0], "xq": flat[:, cols].numpy(), "level_idx": m._level_index(flat, False),
            "noise_idx": None, "mean_idx": m._mean_index(flat)}
    _, _, d = reference_posterior_qbatch(stub.p, stub.h, cand, 2, False, a.numpy(), G.numpy())
    gx = Xb.grad.reshape(-1, Xb.shape[-1])
    np.testing.assert_allclose(gx[:, cols].numpy(), d, rtol=1e-13, atol=1e-15)
    other = [k for k in range(Xb.shape[-1]) if k not in cols]
    assert torch.count_nonzero(gx[:, other]) == 0
    assert all(p.grad is None for p in m.parameters())


def test_backward_restores_the_forward_hyper_parameters():
    m, X = _model("quant")
    Xb = _batch(X, (2, 3)).requires_grad_(True)
    stub = _QBatchEngine(m)
    with m.engine_override(stub):
        post = m.posterior(Xb)
        h0 = dict(stub.h)
        with torch.no_grad():
            m.covar_module.raw_outputscale.add_(0.5)
        m.predict(Xb.detach().reshape(-1, Xb.shape[-1]))  # refactorises for the new outputscale
        assert stub.h["sigma_f2"] != h0["sigma_f2"]
        post.mean.sum().backward()
        assert stub.h["sigma_f2"] == h0["sigma_f2"]


def test_second_derivative_raises():
    m, X = _model("quant")
    Xb = _batch(X, (2, 3)).requires_grad_(True)
    with m.engine_override(_QBatchEngine(m)):
        post = m.posterior(Xb)
        g, = torch.autograd.grad((post.mean ** 2).sum() + post.covariance_matrix.sum(), Xb, create_graph=True)
        with pytest.raises(RuntimeError):
            torch.autograd.grad(g.sum(), Xb)


def test_rsample_with_fixed_base_samples():
    m, X = _model("mixed")
    Xb = _batch(X, (4, 3))
    with m.engine_override(_QBatchEngine(m)):
        post = m.posterior(Xb)
    E = torch.randn(5, 4, 3, generator=torch.Generator().manual_seed(1), dtype=torch.float64)
    draws = post.rsample(torch.Size([5]), base_samples=E)
    assert draws.shape == (5, 4, 3)
    mu, cov = post.mean.numpy(), post.covariance_matrix.numpy()
    for t in range(4):
        L = np.linalg.cholesky(cov[t])
        np.testing.assert_allclose(draws[:, t].numpy(), mu[t][None, :] + E[:, t].numpy() @ L.T, rtol=1e-12, atol=1e-15)
    assert post.rsample(torch.Size([2])).shape == (2, 4, 3)
    with pytest.raises(ValueError, match="base_samples"):
        post.rsample(torch.Size([5]), base_samples=E[:, :2])


def test_rsample_jitters_only_the_singular_block():
    mean = torch.zeros(2, 2, dtype=torch.float64)
    good = torch.tensor([[2.0, 0.5], [0.5, 1.0]], dtype=torch.float64)
    singular = torch.ones(2, 2, dtype=torch.float64)
    E = torch.randn(3, 2, 2, generator=torch.Generator().manual_seed(4), dtype=torch.float64)
    with pytest.warns(NumericalWarning, match="added jitter of 1.0e-08"):
        draws = MultivariateNormal(mean, torch.stack([good, singular])).rsample(torch.Size([3]), base_samples=E)
    np.testing.assert_allclose(draws[:, 0].numpy(), E[:, 0].numpy() @ np.linalg.cholesky(good.numpy()).T, rtol=1e-14)
    L1 = np.linalg.cholesky(singular.numpy() + 1e-8 * np.eye(2))
    np.testing.assert_allclose(draws[:, 1].numpy(), E[:, 1].numpy() @ L1.T, rtol=1e-12)
    with warnings.catch_warnings():
        warnings.simplefilter("error", NumericalWarning)
        MultivariateNormal(mean, torch.stack([good, good])).rsample(torch.Size([3]), base_samples=E)


@pytest.mark.parametrize("kernel", [0, 1, 2])
def test_reference_gradient_matches_central_differences(kernel):
    p = make_problem(30, 3, kernel, dz=2, n_combo=3, n_noise=2, n_mean=2, seed=kernel)
    h = make_hyper(p, seed=1, noise=1e-2)
    q, b = 3, 2
    c = make_candidates(p, b * q, seed=4)
    rng = np.random.default_rng(6)
    gm, gc = rng.standard_normal((b, q)), rng.standard_normal((b, q, q))
    mean, cov, d = reference_posterior_qbatch(p, h, c, q, True, gm, gc)
    eps = 1e-6
    fd = np.zeros_like(d)
    for i in range(b * q):
        for k in range(p["dq"]):
            vals = []
            for s in (1.0, -1.0):
                cs = dict(c)
                cs["xq"] = c["xq"].copy()
                cs["xq"][i, k] += s * eps
                mu_s, cov_s, _ = reference_posterior_qbatch(p, h, cs, q, True)
                vals.append((gm * mu_s).sum() + (gc * cov_s).sum())
            fd[i, k] = (vals[0] - vals[1]) / (2 * eps)
    np.testing.assert_allclose(d, fd, rtol=1e-6, atol=1e-7)
    # the blocks agree with the joint reference of each t-batch alone
    for t in range(b):
        sub = {k: (v[t * q:(t + 1) * q] if isinstance(v, np.ndarray) else v) for k, v in c.items()}
        sub["m"] = q
        mu_t, cov_t = reference_predict_joint(p, h, sub, True)
        np.testing.assert_allclose(cov[t], cov_t, rtol=0, atol=1e-14)
        np.testing.assert_allclose(mean[t], mu_t, rtol=0, atol=1e-14)
