"""Host side of differentiable prediction (GPR.predict with ``x.requires_grad``, GP_Plus.predict_with_grad,
GPR.posterior): the autograd Function that turns the engine's d_mean / d_var into gradients w.r.t. the model's inputs,
driven through a stub engine that answers with the CPU oracle (no GPU needed)."""
import numpy as np
import pytest
import torch

from gpplus_b200._compat import settings
from gpplus_b200.models import GP_Plus
from oracle import gp_oracle as O
from predict_grad_reference import predict_grad as reference_predict_grad


class _OracleEngine:
    """Answers factorize / predict / predict_grad of the model's training set with the CPU references.  With
    ``raw_var_grad`` the variance gradient ignores the clamp (min_var = 0), so that the model layer's own mask is what
    zeroes it."""

    def __init__(self, model, raw_var_grad=False):
        kw = model._engine_kwargs(0)
        xq = kw["xq"] if kw["xq"] is not None else np.zeros((len(kw["y"]), 0))
        self.dq, self.dz, self.n_mean, self.n_pass = xq.shape[1], kw["dz"], kw["n_mean"], kw["n_pass"]
        self.p = {"n": len(kw["y"]), "dq": self.dq, "dz": self.dz, "n_combo": kw["n_combo"], "n_noise": kw["n_noise"],
                  "n_mean": self.n_mean, "kernel": kw["kernel"], "xq": xq, "y": kw["y"], "level_idx": kw["level_idx"],
                  "noise_idx": kw["noise_idx"], "mean_idx": kw["mean_idx"], "n_pass": self.n_pass}
        self.raw_var_grad = raw_var_grad
        self.calls = []

    def factorize(self, hyper):
        self.h = hyper

    def _cand(self, xq, level_idx, noise_idx, mean_idx):
        return {"m": xq.shape[0], "xq": xq, "level_idx": level_idx, "noise_idx": noise_idx, "mean_idx": mean_idx}

    def predict(self, xq, level_idx=None, noise_idx=None, mean_idx=None, include_noise=False, min_var=1e-10):
        self.calls.append("predict")
        return O.predict(self.p, self.h, self._cand(xq, level_idx, noise_idx, mean_idx), include_noise, min_var)

    def predict_grad(self, xq, level_idx=None, noise_idx=None, mean_idx=None, include_noise=False, min_var=1e-10):
        self.calls.append("predict_grad")
        c = self._cand(xq, level_idx, noise_idx, mean_idx)
        mu, var, dm, dv = reference_predict_grad(self.p, self.h, c, include_noise, min_var)
        if self.raw_var_grad:
            dv = reference_predict_grad(self.p, self.h, c, include_noise, 0.0)[3]
        return mu, var, dm, dv


def _model(kind):
    rng = np.random.default_rng(7)
    n = 40
    # columns: 3 quantitative, one categorical (3 levels), the source index last (multi-fidelity models)
    X = np.hstack([rng.standard_normal((n, 3)), rng.integers(0, 3, (n, 1)), rng.integers(0, 2, (n, 1))]).astype(float)
    y = np.sin(X[:, 0]) + 0.3 * X[:, 3] + 0.2 * X[:, 4] + 0.05 * rng.standard_normal(n)
    if kind == "quant":
        m = GP_Plus(torch.tensor(X[:, :3]), torch.tensor(y), dtype=torch.float64,
                    quant_correlation_class="Matern52Kernel")
    else:
        m = GP_Plus(torch.tensor(X), torch.tensor(y), qual_dict={3: 3, 4: 2}, multiple_noise=True,
                    m_gp="multiple_constant", dtype=torch.float64)
    Xq = X[:6, : m.train_inputs[0].shape[1]].copy()
    Xq[:, :3] += 0.3 * rng.standard_normal((6, 3))
    return m, torch.tensor(Xq)


@pytest.mark.parametrize("kind", ["quant", "mixed"])
def test_input_gradient_maps_engine_derivatives_to_columns(kind):
    m, Xq = _model(kind)
    stub = _OracleEngine(m)
    cols = m._quant_columns()
    with m.engine_override(stub):
        x = Xq.clone().requires_grad_(True)
        mean, std = m.predict_with_grad(x, return_std=True, include_noise=True)
        assert stub.calls == ["predict_grad"]
        g_mean, = torch.autograd.grad(mean.sum(), x, retain_graph=True)
        g_std, = torch.autograd.grad(std.sum(), x)
        mean0, std0 = m.predict(Xq, return_std=True, include_noise=True)
    assert torch.equal(mean.detach(), mean0) and torch.equal(std.detach(), std0)
    # the engine's scaled-unit derivatives, by hand: y_std on the mean, y_std / (2 sqrt(var)) on the std
    c = {"m": Xq.shape[0], "xq": Xq[:, cols].numpy(), "level_idx": m._level_index(Xq, False),
         "noise_idx": m._noise_index(Xq), "mean_idx": m._mean_index(Xq)}
    _, var, dm, dv = reference_predict_grad(stub.p, stub.h, c, True, settings.min_variance)
    y_std = float(m.y_std)
    assert np.allclose(g_mean[:, cols].numpy(), y_std * dm, rtol=1e-13, atol=0)
    assert np.allclose(g_std[:, cols].numpy(), y_std * dv / (2.0 * np.sqrt(var))[:, None], rtol=1e-13, atol=0)
    other = [k for k in range(Xq.shape[1]) if k not in cols]
    assert len(other) == (0 if kind == "quant" else 2)
    assert torch.count_nonzero(g_mean[:, other]) == 0 and torch.count_nonzero(g_std[:, other]) == 0
    assert g_mean.dtype == x.dtype and torch.count_nonzero(g_mean[:, cols]) > 0
    # and the whole chain against central differences of predict()
    eps = 1e-6
    for d in cols:
        e = torch.zeros_like(Xq)
        e[:, d] = eps
        with m.engine_override(stub):
            mp, sp = m.predict(Xq + e, return_std=True, include_noise=True)
            mm, sm = m.predict(Xq - e, return_std=True, include_noise=True)
        assert np.allclose(g_mean[:, d].numpy(), ((mp - mm) / (2 * eps)).numpy(), rtol=1e-6, atol=1e-8 * y_std)
        assert np.allclose(g_std[:, d].numpy(), ((sp - sm) / (2 * eps)).numpy(), rtol=1e-6, atol=1e-8 * y_std)


def test_std_gradient_is_zero_where_the_variance_is_clamped(monkeypatch):
    m, Xq = _model("quant")
    stub = _OracleEngine(m, raw_var_grad=True)
    with m.engine_override(stub):
        with torch.no_grad():
            _, std = m.predict(Xq, return_std=True)
        var = (std / m.y_std) ** 2
        s = torch.sort(var).values
        floor = float(0.5 * (s[2] + s[3]))  # three candidates below the floor, three above it
        monkeypatch.setattr(settings, "min_variance", floor)
        x = Xq.clone().requires_grad_(True)
        mean, std = m.predict_with_grad(x, return_std=True)
        g, = torch.autograd.grad(std.sum(), x)
    clamped = (var < floor).numpy()
    assert clamped.sum() == 3
    assert torch.count_nonzero(g[clamped]) == 0 and bool(torch.all(g[~clamped].abs().sum(1) > 0))
    assert np.allclose(((std / m.y_std) ** 2).detach().numpy()[clamped], floor, rtol=1e-12)


def test_second_derivative_raises():
    m, Xq = _model("quant")
    stub = _OracleEngine(m)
    with m.engine_override(stub):
        x = Xq.clone().requires_grad_(True)
        mean, std = m.predict_with_grad(x)
        g, = torch.autograd.grad((mean ** 2).sum() + std.sum(), x, create_graph=True)
        with pytest.raises(RuntimeError):
            torch.autograd.grad(g.sum(), x)


def test_predict_without_a_gradient_never_asks_for_one():
    m, Xq = _model("mixed")
    stub = _OracleEngine(m)
    with m.engine_override(stub):
        m.predict(Xq, return_std=True)
        m.predict_with_grad(Xq)                                  # Xtest does not require a gradient
        m.predict(Xq.clone().requires_grad_(True))               # GP_Plus.predict runs under no_grad
        with torch.no_grad():
            m.predict_with_grad(Xq.clone().requires_grad_(True))
        mean = super(GP_Plus, m).predict(Xq, return_std=False)   # GPR.predict, gradients enabled, plain input
    assert stub.calls == ["predict"] * 5 and not mean.requires_grad


def test_posterior_is_differentiable_in_x():
    m, Xq = _model("quant")
    stub = _OracleEngine(m)
    with m.engine_override(stub):
        x = Xq.clone().requires_grad_(True)
        post = m.posterior(x, observation_noise=False)
        g, = torch.autograd.grad(post.mean.sum(), x)
        _, _, dm, _ = stub.predict_grad(Xq.numpy())
    assert stub.calls == ["predict_grad", "predict_grad"]
    assert np.allclose(g.numpy(), dm, rtol=1e-13, atol=0)
