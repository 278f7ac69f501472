"""GIBBON (max-value entropy search): the quality term against quadrature of the truncated bivariate normal, the
diversity term against slogdet, the CPU reference against central differences, the max-value quartiles against
brentq, and the host side (GPR.gibbon, GPR.sample_max_values, the autograd Function behind them and optimize_gibbon)
driven through a stub engine that answers with the references; no GPU needed."""
import math
import warnings

import numpy as np
import pytest
import torch
from scipy import integrate, optimize, special

from gibbon_reference import (gibbon_block, gibbon_qbatch as reference_gibbon, gumbel_from_quartiles,
                              max_value_quartiles, quality, quartile_bracket)
from gpplus_b200.bayesian_optimizations import optimize_gibbon
from gpplus_b200.models.gpregression import GPR
from oracle import gp_oracle as O
from problems import make_candidates, make_hyper, make_problem
from test_kg import _KgEngine
from test_qbatch_posterior import _batch, _model


def _truncated_variance(v, s2, c, gamma):
    """Var(y | g <= m) for (y, g) jointly normal with Var y = v, Var g = s2, Cov = c and (m - E g) / sd(g) = gamma, by
    quadrature over the truncated bivariate density: g = E g + s u, y = E y + (c / s) u + b w with u, w independent
    standard normals and b^2 = v - c^2 / s2."""
    s = math.sqrt(s2)
    a, b = c / s, math.sqrt(v - c * c / s2)
    dens = lambda w, u: math.exp(-0.5 * (u * u + w * w)) / (2.0 * math.pi)  # noqa: E731
    lo_u = min(gamma, 0.0) - 12.0  # the truncated density below is under e^-72 of its peak
    mom = []
    for k in range(3):  # quadpack's round-off warnings: the tolerance below is asked for, 1e-10 is checked
        warnings.simplefilter("ignore", integrate.IntegrationWarning)
        f = lambda w, u, k=k: (a * u + b * w) ** k * dens(w, u)  # noqa: E731
        val, _ = integrate.nquad(f, [(-12.0, 12.0), (lo_u, gamma)], opts={"epsabs": 0.0, "epsrel": 1e-13, "limit": 200})
        mom.append(val)
    m1, m2 = mom[1] / mom[0], mom[2] / mom[0]
    return m2 - m1 * m1


@pytest.mark.parametrize("rho2", [0.01, 0.5, 0.999])
@pytest.mark.parametrize("gamma", [-6.0, 0.0, 6.0])
def test_quality_is_half_log_variance_ratio(rho2, gamma):
    v, s2, smu = 1.3, 0.7, 0.2
    c = math.sqrt(rho2 * v * s2)
    mv = torch.tensor([smu + gamma * math.sqrt(s2)], dtype=torch.float64)
    args = [torch.tensor([x], dtype=torch.float64) for x in (v, s2, c, smu)]
    q_exact = float(quality(*args, mv, eps=0.0))
    want = 0.5 * math.log(v / _truncated_variance(v, s2, c, gamma))
    assert abs(q_exact - want) <= 1e-10, (q_exact, want)
    q = float(quality(*args, mv))
    if special.ndtr(gamma) > 1e-8:  # botorch's CLAMP_LB is inactive: the formula is the identity
        assert abs(q - want) <= 1e-10
    else:  # Phi(-6) = 9.9e-10 is clamped to 1e-8, which lowers r and the quality
        assert q < q_exact


def test_diversity_is_half_logdet_of_the_correlation_matrix():
    rng = np.random.default_rng(0)
    q = 4
    for jitter_case in (False, True):
        B = rng.standard_normal((q, q))
        V = B @ B.T + 0.1 * np.eye(q)
        noise = np.full((1, q), 0.05)
        if jitter_case:
            V = np.ones((q, q))
            noise = np.zeros((1, q))
        cov = np.zeros((1, 2 * q, 2 * q))  # projected: zero cross block, so every Q_i is 0 and the value is D
        cov[0, :q, :q] = V
        cov[0, q:, q:] = np.eye(q)
        val, _, _, jit = gibbon_block(np.zeros((1, 2 * q)), cov, noise, q, True, [0.3])
        A = V + np.diag(noise[0]) + jit[0] * np.eye(q)
        dA = np.sqrt(np.diag(A))
        sign, logdet = np.linalg.slogdet(A / dA[:, None] / dA[None, :])
        assert sign > 0 and jit[0] == (1e-8 if jitter_case else 0.0)
        if jitter_case:  # ones + j I (condition 4e8): its eigenvalues q + j and j, (q - 1) times, and diagonal 1 + j
            j = jit[0]
            logdet = math.log(q + j) + (q - 1) * math.log(j) - q * math.log1p(j)
        # the factor's pivots of j = 1e-8 carry a rounding of eps / j relative
        tol = 1e-6 if jitter_case else 1e-10 * max(1.0, abs(logdet))
        assert abs(val[0] - 0.5 * logdet) <= tol


def _case(kernel, mixed=False, seed=0):
    if mixed:
        p = make_problem(30, 2, kernel, dz=2, n_combo=3, n_noise=2, n_mean=2, seed=seed, n_pass=3)
    else:
        p = make_problem(30, 3, kernel, seed=seed)
    return p, make_hyper(p, noise=1e-2)


@pytest.mark.parametrize("projected", [False, True])
@pytest.mark.parametrize("maximize", [True, False])
@pytest.mark.parametrize("mixed", [False, True])
def test_reference_gradient_matches_central_differences(mixed, maximize, projected):
    p, h = _case(1, mixed, seed=2)
    q = 2
    q_tot = 2 * q if projected else q
    c = make_candidates(p, 2 * q_tot, seed=5)
    mv = np.array([0.9, 1.1, 1.4]) * (1.0 if maximize else -0.2)
    v, d, jit = reference_gibbon(p, h, c, q, projected, mv, maximize)
    assert np.all(np.isfinite(v)) and (jit == 0).all()
    eps = 1e-6
    fd = np.zeros_like(d)
    for r in range(d.shape[0]):
        for k in range(p["dq"]):
            vals = []
            for s in (1.0, -1.0):
                cc = dict(c)
                cc["xq"] = np.array(c["xq"])
                cc["xq"][r, k] += s * eps
                vals.append(reference_gibbon(p, h, cc, q, projected, mv, maximize, jit)[0].sum())
            fd[r, k] = (vals[0] - vals[1]) / (2 * eps)
    assert np.abs(d).max() > 1e-3
    np.testing.assert_allclose(d, fd, rtol=1e-5, atol=1e-8)


@pytest.mark.parametrize("m", [1, 50, 20000])
@pytest.mark.parametrize("maximize", [True, False])
def test_quartiles_match_brentq_and_the_gumbel_fit(m, maximize):
    rng = np.random.default_rng(m)
    mean = rng.standard_normal(m)
    var = rng.uniform(0.01, 0.5, m)
    qs, lo, hi = max_value_quartiles(mean, var, maximize)
    _, _, smu, sd = quartile_bracket(mean, var, maximize)
    for y, p in zip(qs, (0.25, 0.5, 0.75)):
        f = lambda t: float(torch.special.log_ndtr((t - smu) / sd).sum()) - math.log(p)  # noqa: E731
        root = optimize.brentq(f, lo, hi, xtol=1e-15 * (hi - lo), rtol=4 * np.finfo(float).eps)
        assert abs(y - root) <= 1e-12 * (hi - lo)
    alpha, beta = gumbel_from_quartiles(*qs)  # fitted at the median exactly, at the other two by their spread
    assert beta > 0 and abs(math.exp(-math.exp(-(qs[1] - alpha) / beta)) - 0.5) <= 1e-14


def test_gumbel_fit_round_trip():
    for alpha, beta in ((1.3, 0.4), (-2.0, 3e-3)):
        p = np.array([0.25, 0.5, 0.75])
        qs = alpha - beta * np.log(-np.log(p))
        a, b = gumbel_from_quartiles(*qs)
        assert math.isclose(a, alpha, rel_tol=1e-14, abs_tol=1e-14) and math.isclose(b, beta, rel_tol=1e-12)
        np.testing.assert_allclose(np.exp(-np.exp(-(qs - a) / b)), p, rtol=0, atol=1e-13)


def test_quartile_bracket_widens_for_many_candidates():
    mean, var = np.zeros(2_000_000), np.ones(2_000_000)
    lo, hi, _, _ = quartile_bracket(mean, var)
    assert hi > 5.0 and math.isclose(lo, -5.0)
    qs, _, _ = max_value_quartiles(mean, var)
    assert lo < qs[0] < qs[1] < qs[2] < hi


# ---- the host side through a stub engine ----


class _GibbonEngine(_KgEngine):
    """Adds gibbon_qbatch and max_value_quartiles, answered by the references; records every gibbon_qbatch call."""

    def __init__(self, model):
        super().__init__(model)
        self.gb = []

    def gibbon_qbatch(self, xq, q, max_values, projected=False, maximize=True, want_grad=True, level_idx=None,
                      noise_idx=None, mean_idx=None):
        self.calls.append("gibbon_qbatch")
        self.gb.append(dict(xq=xq, q=q, mv=np.asarray(max_values), projected=projected, maximize=maximize,
                            want_grad=want_grad, level_idx=level_idx, noise_idx=noise_idx, mean_idx=mean_idx))
        v, d, jit = reference_gibbon(self.p, self.h, self._cand(xq, level_idx, noise_idx, mean_idx), q, projected,
                                     max_values, maximize)
        return v, (d if want_grad else None), jit

    def max_value_quartiles(self, xq, level_idx=None, mean_idx=None, maximize=True):
        self.calls.append("max_value_quartiles")
        mean, var = O.predict(self.p, self.h, self._cand(xq, level_idx, None, mean_idx), False, 1e-8)
        return max_value_quartiles(mean, var, maximize)[0]


def _scaled(stub, a):
    return reference_gibbon(stub.p, stub.h, stub._cand(a["xq"], a["level_idx"], a["noise_idx"], a["mean_idx"]),
                            a["q"], a["projected"], a["mv"], a["maximize"])


@pytest.mark.parametrize("maximize", [True, False])
@pytest.mark.parametrize("projected", [False, True])
def test_values_max_value_units_and_projection_gradient_fold(projected, maximize):
    m, X = _model("mixed")
    q = 2
    Xb = _batch(X, (2, 3, q)).requires_grad_(True)
    stub = _GibbonEngine(m)
    mv = torch.tensor([8.5, 9.0, 9.7]) if maximize else torch.tensor([1.0, 0.5])
    sgn = 1.0 if maximize else -1.0
    tfc = {4: 0.0} if projected else None
    with m.engine_override(stub):
        v = m.gibbon(Xb, mv, maximize=maximize, target_fixed_columns=tfc)
        v.sum().backward()
    a = stub.gb[-1]
    assert a["want_grad"] and a["q"] == q and a["projected"] is projected and a["maximize"] is maximize
    np.testing.assert_allclose(a["mv"], sgn * (mv.double().numpy() - float(m.y_min)) / float(m.y_std), rtol=1e-15)
    rows = Xb.detach().reshape(6, q, -1)
    if projected:
        tgt = rows.clone()
        tgt[:, :, 4] = 0.0
        rows = torch.cat([rows, tgt], 1)
    np.testing.assert_array_equal(a["xq"], rows.reshape(-1, X.shape[1])[:, m._quant_columns()].numpy())
    np.testing.assert_array_equal(a["noise_idx"], m._noise_index(rows.reshape(-1, X.shape[1])))
    v_sc, d_sc, _ = _scaled(stub, a)
    np.testing.assert_allclose(v.detach().numpy().reshape(-1), v_sc, rtol=1e-13)
    cols = m._quant_columns()
    d_sc = d_sc.reshape(6, -1, len(cols))
    want = d_sc[:, :q] + d_sc[:, q:] if projected else d_sc
    g = Xb.grad.reshape(6, q, -1)
    np.testing.assert_allclose(g[:, :, cols].numpy(), want, rtol=1e-12, atol=1e-14)
    assert bool((g[:, :, [c for c in range(X.shape[1]) if c not in cols]] == 0).all())
    assert v.shape == (2, 3) and v.dtype == torch.float64


def test_gradient_with_a_quantitative_target_column_matches_central_differences():
    """A continuous fidelity column held at its target value on the target rows (botorch's
    project_to_target_fidelity): the target rows do not move with X in that column, so its gradient comes from the
    actual rows alone, while the other quantitative columns fold both copies."""
    m, X = _model("mixed")
    Xb = _batch(X, (2, 2)).requires_grad_(True)
    P = _batch(X, (1,), seed=9)
    stub = _GibbonEngine(m)
    mv = torch.tensor([8.5, 9.7])
    tfc = {2: 0.4, 4: 0.0}
    with m.engine_override(stub):
        v = m.gibbon(Xb, mv, target_fixed_columns=tfc, X_pending=P)
        v.sum().backward()
        _, d_sc, _ = _scaled(stub, stub.gb[0])
        assert np.abs(d_sc.reshape(2, 6, 3)[:, 3:5, 2]).max() > 1e-3  # the target rows' own gradient in column 2
        eps = 1e-6
        fd = torch.zeros_like(Xb)
        with torch.no_grad():
            for t in range(2):
                for i in range(2):
                    for c in m._quant_columns():
                        vals = []
                        for s_ in (1.0, -1.0):
                            Xp = Xb.detach().clone()
                            Xp[t, i, c] += s_ * eps
                            vals.append(float(m.gibbon(Xp, mv, target_fixed_columns=tfc, X_pending=P).sum()))
                        fd[t, i, c] = (vals[0] - vals[1]) / (2 * eps)
    cols = m._quant_columns()
    print("gradient vs central differences %.2e" % float((Xb.grad[..., cols] - fd[..., cols]).abs().max()))
    np.testing.assert_allclose(Xb.grad[..., cols].numpy(), fd[..., cols].numpy(), rtol=1e-5, atol=1e-7)


def test_pending_points_are_subtracted_and_get_no_gradient():
    m, X = _model("mixed")
    Xb = _batch(X, (3, 1)).requires_grad_(True)
    P = _batch(X, (2,), seed=9)
    stub = _GibbonEngine(m)
    mv = torch.tensor([8.5, 9.7])
    tfc = {4: 0.0}
    with m.engine_override(stub):
        v = m.gibbon(Xb, mv, target_fixed_columns=tfc, X_pending=P)
        v.sum().backward()
        joint = m.gibbon(torch.cat([Xb.detach(), P.expand(3, 2, -1)], 1), mv, target_fixed_columns=tfc)
        alone = m.gibbon(P[None], mv, target_fixed_columns=tfc)
        with torch.no_grad():
            assert stub.gb[0]["q"] == 3 and not stub.gb[1]["want_grad"] and stub.gb[1]["q"] == 2
    np.testing.assert_allclose(v.detach().numpy(), (joint - alone).detach().numpy(), rtol=1e-13, atol=1e-14)
    a = stub.gb[0]
    _, d_sc, _ = _scaled(stub, a)
    cols = m._quant_columns()
    d_sc = d_sc.reshape(3, 6, len(cols))
    np.testing.assert_allclose(Xb.grad[:, :, cols].numpy(), d_sc[:, :1] + d_sc[:, 3:4], rtol=1e-12, atol=1e-14)


def test_cost_divides_the_gain_by_the_rows_summed_cost():
    m, X = _model("mixed")
    Xb = _batch(X, (4, 2))
    P = _batch(X, (1,), seed=3)
    stub = _GibbonEngine(m)
    mv = torch.tensor([9.0])
    with m.engine_override(stub), torch.no_grad():
        v = m.gibbon(Xb, mv, X_pending=P)
        vc = m.gibbon(Xb, mv, X_pending=P, cost_by_source={0: 10.0, 1: 1.5})
        vl = m.gibbon(Xb, mv, X_pending=P, cost_by_source=[10.0, 1.5])
    src = Xb[..., -1]
    total = (10.0 * (src == 0) + 1.5 * (src == 1)).sum(-1)
    np.testing.assert_allclose(vc.numpy(), (v / total).numpy(), rtol=1e-14)
    assert torch.equal(vc, vl)


def test_argument_errors():
    m, X = _model("mixed")
    stub = _GibbonEngine(m)
    Xb = _batch(X, (2, 2))
    cands = _batch(X, (20,))
    with m.engine_override(stub):
        for args, kw, match in (((Xb[0, 0], [1.0]), {}, "expects X"),
                                ((Xb, []), {}, "max values"),
                                ((_batch(X, (1, 65)), [1.0]), dict(target_fixed_columns={4: 0.0}), "outside"),
                                ((Xb, [1.0]), dict(X_pending=_batch(X, (127,))), "outside")):
            with pytest.raises(ValueError, match=match):
                m.gibbon(*args, **kw)
        for kw, match in ((dict(method="exact"), "method"), (dict(num_samples=0), "num_samples")):
            with pytest.raises(ValueError, match=match):
                m.sample_max_values(cands, **kw)
        with pytest.raises(ValueError, match="candidate_set"):
            m.sample_max_values(cands[None])
        bounds = np.array([[-1.0, -0.5, 0.0], [1.0, 0.5, 2.0]])
        fixed = {3: 1.0, 4: 0.0}
        for kw, match in ((dict(sources=[0, 1], sequential=False), "sequential"),
                          (dict(sources=[]), "empty"), (dict(fixed_columns={3: 1.0}), "need fixed_columns")):
            args = dict(fixed_columns=fixed)
            args.update(kw)
            with pytest.raises(ValueError, match=match):
                optimize_gibbon(m, bounds, 1, [9.0], **args)
        with pytest.raises(ValueError, match="q must be"):
            optimize_gibbon(m, bounds, 0, [9.0], fixed_columns=fixed)
    mq, Xq = _model("quant")
    with mq.engine_override(_GibbonEngine(mq)):
        with pytest.raises(ValueError, match="not a quantitative one"):
            optimize_gibbon(mq, np.array([[-1.0] * 3, [1.0] * 3]), 1, [9.0], sources=[0, 1])
    assert "gibbon_qbatch" not in stub.calls


def test_sample_max_values_gumbel_is_seeded_and_in_y_units():
    m, X = _model("quant")
    stub = _GibbonEngine(m)
    cands = _batch(X, (40,))
    with m.engine_override(stub):
        for maximize in (True, False):
            s1 = m.sample_max_values(cands, 16, maximize=maximize, seed=3)
            s2 = m.sample_max_values(cands, 16, maximize=maximize, seed=3)
            s3 = m.sample_max_values(cands, 16, maximize=maximize, seed=4)
            assert torch.equal(s1, s2) and not torch.equal(s1, s3) and s1.shape == (16,)
            xq = cands[:, m._quant_columns()].numpy()
            qs = stub.max_value_quartiles(xq, maximize=maximize)
            alpha, beta = gumbel_from_quartiles(*qs)
            u = torch.rand(16, generator=torch.Generator().manual_seed(3), dtype=torch.float64)
            want = alpha - beta * torch.log(-torch.log(u))
            sgn = 1.0 if maximize else -1.0
            np.testing.assert_allclose(s1.numpy(), float(m.y_min) + sgn * float(m.y_std) * want.numpy(), rtol=1e-14)
            with torch.no_grad():
                mu = GPR.predict(m, cands)
            if maximize:  # the median of the maximum lies above the largest mean
                assert float(s1.median()) > float(mu.max()) - 1e-9
            else:
                assert float(s1.median()) < float(mu.min()) + 1e-9


def test_sequential_equals_joint_at_q1_and_sources_pick_by_gain_per_cost():
    m, X = _model("mixed")
    stub = _GibbonEngine(m)
    bounds = np.array([[-1.0, -0.5, 0.0], [1.0, 0.5, 2.0]])
    mv = [9.2, 9.6]
    args = dict(fixed_columns={3: 1.0, 4: 0.0}, num_restarts=2, raw_samples=8, options={"maxiter": 4}, seed=1)
    with m.engine_override(stub):
        Xs, vs = optimize_gibbon(m, bounds, 1, mv, sequential=True, **args)
        Xj, vj = optimize_gibbon(m, bounds, 1, mv, sequential=False, **args)
        assert torch.equal(Xs, Xj) and vs == vj and Xs.shape == (1, 5)
        tfc = {4: 0.0}
        for cost in ({0: 10.0, 1: 1.0}, {0: 1.0, 1: 50.0}):
            Xc, vc = optimize_gibbon(m, bounds, 2, mv, target_fixed_columns=tfc, cost_by_source=cost, sources=[0, 1],
                                     **args)
            assert Xc.shape == (2, 5) and bool((Xc[:, 3] == 1.0).all()) and np.isfinite(vc)
            with torch.no_grad():
                assert vc == float(m.gibbon(Xc[None], mv, target_fixed_columns=tfc, cost_by_source=cost)[0])
            # the first pick: the better of the two single-source searches, by gain per unit cost
            per_src = []
            for s in (0, 1):
                a = dict(args)
                a["fixed_columns"] = {3: 1.0, 4: float(s)}
                Xo, _ = optimize_gibbon(m, bounds, 1, mv, target_fixed_columns=tfc, cost_by_source=cost, **a)
                with torch.no_grad():
                    per_src.append((float(m.gibbon(Xo[None], mv, target_fixed_columns=tfc, cost_by_source=cost)[0]),
                                    Xo[0]))
            best = per_src[1] if per_src[1][0] > per_src[0][0] else per_src[0]
            assert torch.equal(Xc[0], best[1])
            q_lo = Xc[:, :3] >= torch.tensor(bounds[0])
            assert bool(q_lo.all()) and bool((Xc[:, :3] <= torch.tensor(bounds[1])).all())
