"""Host side of Monte-Carlo batch acquisition (GPR.acquisition_qbatch, the autograd Function behind it and
bayesian_optimizations.optimize_acquisition_qbatch), driven through a stub engine that answers with the CPU reference
(tests/qacq_reference.py); no GPU needed."""
import warnings

import numpy as np
import pytest
import torch

from gpplus_b200 import _engine
from gpplus_b200._compat import NumericalWarning
from gpplus_b200.bayesian_optimizations import optimize_acquisition_qbatch
from gpplus_b200.models.gpregression import sobol_normal_samples
from qacq_reference import acq_qbatch as reference_acq, mc_utility
from qbatch_posterior_reference import posterior_qbatch as reference_posterior_qbatch
from test_qbatch_posterior import _QBatchEngine, _batch, _model


class _AcqEngine(_QBatchEngine):
    """Adds acquisition_qbatch, answered by the reference, with an optional forced jitter or error."""

    jitter = None
    error = None

    def acquisition_qbatch(self, xq, q_tot, kind, base_samples, best_f=0.0, beta=0.0, n_baseline=0, maximize=True,
                           want_grad=True, level_idx=None, noise_idx=None, mean_idx=None, include_noise=False):
        self.calls.append("acquisition_qbatch")
        self.acq = dict(xq=xq, q_tot=q_tot, kind=kind, E=np.asarray(base_samples), best_f=best_f, beta=beta,
                        n_baseline=n_baseline, maximize=maximize, want_grad=want_grad, level_idx=level_idx,
                        noise_idx=noise_idx, mean_idx=mean_idx, include_noise=include_noise)
        if self.error is not None:
            raise self.error
        cand = self._cand(xq, level_idx, noise_idx, mean_idx)
        b = xq.shape[0] // q_tot
        jit = None if self.jitter is None else np.asarray(self.jitter)[:b]
        v, d, jit = reference_acq(self.p, self.h, cand, q_tot, kind, base_samples, best_f, beta, n_baseline, maximize,
                                  include_noise, jit)
        return v, (d if want_grad else None), jit


def _scaled_reference(stub, kind, **kw):
    a = stub.acq
    cand = stub._cand(a["xq"], a["level_idx"], a["noise_idx"], a["mean_idx"])
    return reference_acq(stub.p, stub.h, cand, a["q_tot"], kind, a["E"], **kw)


@pytest.mark.parametrize("maximize", [True, False])
@pytest.mark.parametrize("kind", ["qEI", "qUCB"])
def test_units_of_values_best_f_and_gradients(kind, maximize):
    m, X = _model("quant")
    Xb = _batch(X, (3, 2, 4)).requires_grad_(True)
    stub = _AcqEngine(m)
    y_min, y_std = float(m.y_min), float(m.y_std)
    best_f = y_min + 0.6 * y_std
    kw = dict(best_f=best_f) if kind == "qEI" else dict(beta=0.7)
    with m.engine_override(stub):
        v = m.acquisition_qbatch(Xb, kind, maximize=maximize, num_samples=64, **kw)
        v.sum().backward()
    assert v.shape == (3, 2) and v.dtype == torch.float64
    a = stub.acq
    assert a["want_grad"] and a["maximize"] == maximize and a["E"].shape == (64, 4)
    np.testing.assert_array_equal(a["E"], sobol_normal_samples(64, 4, 0).numpy())
    sk = _engine.QACQ_EI if kind == "qEI" else _engine.QACQ_UCB
    assert a["kind"] == sk
    if kind == "qEI":
        assert a["best_f"] == pytest.approx(0.6, rel=1e-14)
    v_sc, d_sc, _ = _scaled_reference(stub, sk, best_f=a["best_f"], beta=a["beta"], maximize=maximize)
    sgn = 1.0 if maximize else -1.0
    want = y_std * v_sc if kind == "qEI" else sgn * y_min + y_std * v_sc
    np.testing.assert_allclose(v.detach().reshape(-1).numpy(), want, rtol=1e-13)
    np.testing.assert_allclose(Xb.grad.reshape(-1, 3).numpy(), y_std * d_sc, rtol=1e-12, atol=1e-14)


def test_no_gradient_requested_without_requires_grad():
    m, X = _model("quant")
    stub = _AcqEngine(m)
    with m.engine_override(stub):
        v = m.acquisition_qbatch(_batch(X, (2, 3)), "qUCB", beta=1.0, num_samples=16)
        x = _batch(X, (2, 3)).requires_grad_(True)
        with torch.no_grad():
            m.acquisition_qbatch(x, "qUCB", beta=1.0, num_samples=16)
    assert not v.requires_grad and stub.acq["want_grad"] is False


def test_baseline_rows_and_level_ranking():
    m, X = _model("mixed")
    Xb = _batch(X, (2, 3))
    base = _batch(X, (4,), seed=9)
    stub = _AcqEngine(m)
    with m.engine_override(stub):
        m.acquisition_qbatch(Xb, "qNEI", X_baseline=base, num_samples=8)
    a = stub.acq
    assert a["q_tot"] == 7 and a["n_baseline"] == 4 and a["E"].shape == (8, 7)
    rows = torch.cat([Xb, base.expand(2, 4, base.shape[-1])], dim=1).reshape(-1, Xb.shape[-1])
    cols = m._quant_columns()
    np.testing.assert_array_equal(a["xq"], rows[:, cols].numpy())
    # categorical levels ranked against train, every row of X and the baseline
    assert np.array_equal(a["level_idx"], m._level_index(rows, False))
    assert np.array_equal(a["mean_idx"], m._mean_index(rows))


def test_arguments_per_kind():
    m, X = _model("quant")
    Xb = _batch(X, (2, 3))
    with m.engine_override(_AcqEngine(m)):
        with pytest.raises(ValueError, match="best_f"):
            m.acquisition_qbatch(Xb, "qEI")
        with pytest.raises(ValueError, match="X_baseline"):
            m.acquisition_qbatch(Xb, "qNEI")
        with pytest.raises(ValueError, match="beta"):
            m.acquisition_qbatch(Xb, "qUCB")
        with pytest.raises(ValueError, match="kind"):
            m.acquisition_qbatch(Xb, "qPI", best_f=0.0)
        with pytest.raises(ValueError, match="exceeds"):
            m.acquisition_qbatch(_batch(X, (1, 120)), "qNEI", X_baseline=_batch(X, (9,)))
        with pytest.raises(ValueError, match="base_samples"):
            m.acquisition_qbatch(Xb, "qEI", best_f=1.0, base_samples=torch.zeros(4, 2))


def test_jitter_warning_and_error_mapping():
    m, X = _model("quant")
    Xb = _batch(X, (3, 2))
    stub = _AcqEngine(m)
    with m.engine_override(stub):
        stub.jitter = np.array([0.0, 1e-7, 0.0])
        with pytest.warns(NumericalWarning, match="1.0e-07"):
            m.acquisition_qbatch(Xb, "qEI", best_f=6.0, num_samples=8)
        stub.jitter = np.zeros(3)
        with warnings.catch_warnings():
            warnings.simplefilter("error", NumericalWarning)
            m.acquisition_qbatch(Xb, "qEI", best_f=6.0, num_samples=8)
        for err in (_engine.NotPSDError("not p.d."), _engine.NanError("nan")):
            stub.error = err
            with pytest.raises(type(err)):
                m.acquisition_qbatch(Xb, "qEI", best_f=6.0, num_samples=8)


def test_engine_status_codes_map_to_the_gpytorch_errors():
    with pytest.raises(_engine.NotPSDError):
        _engine._raise(_engine.GPP_ERR_NOT_PD, "gpp_acq_qbatch")
    with pytest.raises(_engine.NanError):
        _engine._raise(_engine.GPP_ERR_NAN, "gpp_acq_qbatch")


def test_backward_scales_each_t_batch_by_its_upstream_gradient():
    m, X = _model("mixed")
    Xb = _batch(X, (4, 3), seed=11).requires_grad_(True)
    stub = _AcqEngine(m)
    w = torch.tensor([0.5, -2.0, 0.0, 3.0], dtype=torch.float64)
    with m.engine_override(stub):
        v = m.acquisition_qbatch(Xb, "qEI", best_f=float(m.y_min) + 0.5 * float(m.y_std), num_samples=32)
        (w * v).sum().backward()
        n_calls = stub.calls.count("acquisition_qbatch")
    assert n_calls == 1  # the backward makes no engine call
    v_sc, d_sc, _ = _scaled_reference(stub, _engine.QACQ_EI, best_f=stub.acq["best_f"])
    cols = m._quant_columns()
    g = Xb.grad
    want = float(m.y_std) * w[:, None, None].numpy() * d_sc.reshape(4, 3, len(cols))
    np.testing.assert_allclose(g[:, :, cols].numpy(), want, rtol=1e-12, atol=1e-14)
    other = [k for k in range(Xb.shape[-1]) if k not in cols]
    assert torch.count_nonzero(g[:, :, other]) == 0


def test_reference_utility_gradient_matches_central_differences():
    rng = np.random.default_rng(1)
    b, q = 2, 4
    A = rng.standard_normal((b, q, q))
    cov = A @ A.transpose(0, 2, 1) + 0.5 * np.eye(q)
    mean = rng.standard_normal((b, q))
    E = rng.standard_normal((16, q))
    for kind, kw in ((0, dict(best_f=0.3)), (1, dict(n_baseline=2)), (2, dict(beta=0.8))):
        _, gm, gc, _ = mc_utility(mean, cov, E, kind, **kw)
        eps = 1e-6
        for t, i, j in ((0, 1, 1), (1, 3, 0), (0, 2, 3)):
            cp, cm = cov.copy(), cov.copy()
            for c in (cp, cm):
                s = eps if c is cp else -eps
                c[t, i, j] += s
                if i != j:
                    c[t, j, i] += s
            fd = (mc_utility(mean, cp, E, kind, **kw)[0].sum() - mc_utility(mean, cm, E, kind, **kw)[0].sum()) / (2 * eps)
            an = gc[t, i, j] + (gc[t, j, i] if i != j else 0.0)
            assert abs(fd - an) <= 1e-6 * max(1.0, abs(an)), (kind, t, i, j, fd, an)
        mp = mean.copy()
        mp[1, 2] += eps
        mm = mean.copy()
        mm[1, 2] -= eps
        fd = (mc_utility(mp, cov, E, kind, **kw)[0].sum() - mc_utility(mm, cov, E, kind, **kw)[0].sum()) / (2 * eps)
        assert abs(fd - gm[1, 2]) <= 1e-6


def _opt_model():
    m, X = _model("mixed")
    return m, X


def test_optimizer_screens_keeps_bounds_and_fixed_columns():
    m, X = _opt_model()
    stub = _AcqEngine(m)
    seen = []
    orig = m.acquisition_qbatch

    def spy(Xc, kind, **kw):
        seen.append(Xc.detach().clone())
        return orig(Xc, kind, **kw)

    m.acquisition_qbatch = spy
    bounds = np.array([[-1.0, -0.5, 0.0], [1.0, 0.5, 2.0]])
    fixed = {3: 1.0, 4: 0.0}
    best_f = float(m.y_min) + 0.7 * float(m.y_std)
    with m.engine_override(stub):
        X1, v1 = optimize_acquisition_qbatch(m, bounds, 2, "qEI", fixed_columns=fixed, num_restarts=3, raw_samples=16,
                                             options={"maxiter": 5}, seed=4, best_f=best_f, num_samples=32)
        raw = seen[0]
        with torch.no_grad():
            v_raw = orig(raw, "qEI", best_f=best_f, base_samples=sobol_normal_samples(32, 2, 4))
        X2, v2 = optimize_acquisition_qbatch(m, bounds, 2, "qEI", fixed_columns=fixed, num_restarts=3, raw_samples=16,
                                             options={"maxiter": 5}, seed=4, best_f=best_f, num_samples=32)
    assert raw.shape == (16, 2, 5)
    starts = seen[1]  # the first L-BFGS-B evaluation is at the screened starts
    order = np.lexsort((np.arange(16), -v_raw.numpy()))[:3]
    assert torch.equal(starts, raw[torch.as_tensor(order)])
    for Xc in seen + [X1[None]]:
        q = Xc[..., :3]
        assert bool((q >= torch.tensor(bounds[0])).all()) and bool((q <= torch.tensor(bounds[1])).all())
        assert bool((Xc[..., 3] == 1.0).all()) and bool((Xc[..., 4] == 0.0).all())
    assert X1.shape == (2, 5)
    assert torch.equal(X1, X2) and v1 == v2
    with pytest.raises(ValueError, match="fixed_columns"):
        optimize_acquisition_qbatch(m, bounds, 2, "qEI", best_f=best_f)
