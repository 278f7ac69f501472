"""gpp_kg_qbatch on the B200: one-shot knowledge-gradient values and input gradients against torch on the engine's own
t-batch posteriors and against the dense CPU reference (tests/kg_reference.py), bitwise identities (repeated,
values-only, sub-ranges across chunk boundaries, device-resident), the zero-sample limit, central differences, the
per-t-batch jitter, the untouched handle, argument and status codes, and cost-aware multi-fidelity KG end to end."""
import numpy as np
import pytest
import torch

from kg_reference import kg_block, kg_qbatch as reference_kg
from problems import engine_kwargs, make_candidates, make_hyper, make_problem
from qacq_reference import ladder_jitter

pytestmark = pytest.mark.gpu

VAL_TOL_ENGINE = 1e-9  # |v - v_torch| on the engine's own blocks, scaled units
VAL_TOL_DENSE = 1e-8   # |v - v_ref| against the dense CPU reference, scaled units
GRAD_TOL = 1e-7        # |d - d_ref| relative to the largest |d_ref|


def _engine(p, fp64=None):
    from gpplus_b200 import _engine as E
    prev = E.set_fp64_mode(fp64) if fp64 is not None else None
    try:
        eng = E.Engine(**engine_kwargs(p))
    finally:
        if fp64 is not None:
            E.set_fp64_mode(prev)
    if fp64 is not None:
        assert eng.fp64_mode() == fp64
    return eng


def _kw(c):
    return dict(level_idx=c["level_idx"], noise_idx=c["noise_idx"], mean_idx=c["mean_idx"])


def _base(nf, q, seed=0):
    from gpplus_b200.models.gpregression import sobol_normal_samples
    return np.ascontiguousarray(sobol_normal_samples(nf, q, seed).numpy())


def _check(p, h, c, q, nf, fp64=None, maximize=True, dense=True):
    q_tot = q + nf
    b = c["m"] // q_tot
    kw = _kw(c)
    E = _base(nf, q, seed=q_tot)
    eng = _engine(p, fp64)
    try:
        eng.factorize(h)
        mu0, var0 = eng.predict(c["xq"], min_var=-np.inf, **kw)
        alpha0, stats0 = eng.fetch("alpha"), eng.stats()
        mean, cov = eng.posterior_qbatch(c["xq"], q_tot, include_noise=True, **kw)
        v, d, jit = eng.kg_qbatch(c["xq"], q, nf, E, maximize=maximize, **kw)
        v1, d1, jit1 = eng.kg_qbatch(c["xq"], q, nf, E, maximize=maximize, **kw)
        v0, none, jit0 = eng.kg_qbatch(c["xq"], q, nf, E, maximize=maximize, want_grad=False, **kw)
        vt, gm, gc, _ = kg_block(mean, cov, q, E, maximize, jit)
        d_eng = eng.posterior_qbatch_grad(c["xq"], q_tot, gm, gc, include_noise=True, **kw)
        mu1, var1 = eng.predict(c["xq"], min_var=-np.inf, **kw)
        assert np.array_equal(eng.fetch("alpha"), alpha0) and np.array_equal(mu1, mu0) and np.array_equal(var1, var0)
        assert eng.stats() == stats0
    finally:
        eng.close()
    assert v.shape == (b,) and d.shape == (b * q_tot, p["dq"]) and jit.shape == (b,) and none is None
    assert np.all(np.isfinite(v)) and np.all(np.isfinite(d))
    assert np.array_equal(v, v1) and np.array_equal(d, d1) and np.array_equal(jit, jit1), "repeated calls differ"
    assert np.array_equal(v0, v) and np.array_equal(jit0, jit), "values-only differs from the gradient call"
    np.testing.assert_array_equal(jit, ladder_jitter(torch.from_numpy(cov[:, :q, :q])).numpy())
    cond = float(np.max(np.linalg.cond(cov[:, :q, :q] + jit[:, None, None] * np.eye(q))))
    verr = float(np.max(np.abs(v - vt)))
    scale = max(1.0, float(np.max(np.abs(d_eng), initial=0.0)))
    derr = float(np.max(np.abs(d - d_eng), initial=0.0)) / scale
    print("q=%d F=%d b=%d cond %.1e jitter %.0e: engine blocks value %.2e d_xq %.2e"
          % (q, nf, b, cond, float(jit.max()), verr, derr))
    assert cond < 1e6, cond
    assert verr <= VAL_TOL_ENGINE, verr
    assert derr <= GRAD_TOL, derr
    if dense:
        rv, rd, _ = reference_kg(p, h, c, q, nf, E, maximize, jit)
        rverr = float(np.max(np.abs(v - rv)))
        rderr = float(np.max(np.abs(d - rd), initial=0.0)) / max(1.0, float(np.max(np.abs(rd), initial=0.0)))
        print("   dense reference: value %.2e d_xq %.2e" % (rverr, rderr))
        assert rverr <= VAL_TOL_DENSE, rverr
        assert rderr <= GRAD_TOL, rderr
    return v, d, jit


@pytest.mark.parametrize("kernel", [0, 1, 2])
@pytest.mark.parametrize("q,nf", [(1, 1), (1, 64), (4, 16), (8, 64), (64, 64), (127, 1), (1, 127)])
def test_kernels_and_batch_shapes(kernel, q, nf):
    p = make_problem(300, 4, kernel, seed=kernel + 1)
    b = max(2, 384 // (q + nf))
    _check(p, make_hyper(p, seed=3, noise=1e-2), make_candidates(p, b * (q + nf), seed=q + nf), q, nf,
           maximize=kernel != 1)


@pytest.mark.parametrize("n_pass", [1, 3])
def test_latent_map_and_ensemble(n_pass):
    p = make_problem(260, 3, 2, dz=2, n_combo=6, n_pass=n_pass, seed=11)
    _check(p, make_hyper(p, seed=4, noise=1e-2), make_candidates(p, 40 * 7, seed=6), 3, 4)


@pytest.mark.parametrize("maximize", [True, False])
def test_noise_groups_and_means(maximize):
    p = make_problem(300, 5, 1, dz=2, n_combo=4, n_noise=3, n_mean=3, zero_mean_group=True, seed=12)
    _check(p, make_hyper(p, seed=5, noise=1e-2), make_candidates(p, 37 * 9, seed=7), 4, 5, maximize=maximize)


@pytest.mark.parametrize("dq", [0, 32])
def test_input_widths(dq):
    if dq == 0:
        p = make_problem(200, 0, 0, dz=2, n_combo=5, seed=14)
        h = make_hyper(p, seed=7, noise=1e-2)
    else:
        p = make_problem(400, 32, 2, seed=13)
        h = make_hyper(p, seed=6, noise=1e-2, w_scale=0.02)
    _check(p, h, make_candidates(p, 30 * 6, seed=8), 2, 4)


@pytest.mark.parametrize("fp64", ["dmma", "int8"])
def test_int8_sliced_factor(fp64):
    from gpplus_b200 import _engine as E
    p = make_problem(3200, 4, 2, seed=15)
    _check(p, make_hyper(p, seed=8, noise=1e-2), make_candidates(p, 40 * 12, seed=10), 4, 8,
           fp64=E.FP64_DMMA if fp64 == "dmma" else E.FP64_INT8)


def test_other_batches_and_chunk_split_do_not_matter():
    """N = 3200, dq = 32, q_tot = 3: chunks of 163 tiles of 42 t-batches, so 13 709 t-batches take three chunks.  Any
    run of t-batches called alone gives bitwise the full call's values, jitters and gradients, and so do
    device-resident inputs and outputs."""
    p = make_problem(3200, 32, 2, n_noise=2, n_mean=2, seed=18)
    h = make_hyper(p, seed=10, noise=1e-3, w_scale=0.02)
    q, nf, b = 1, 2, 163 * 42 * 2 + 17
    c = make_candidates(p, b * (q + nf), seed=19)
    kw = _kw(c)
    Eb = _base(nf, q, seed=5)
    eng = _engine(p)
    try:
        eng.factorize(h)
        v, d, jit = eng.kg_qbatch(c["xq"], q, nf, Eb, **kw)
        for lo, hi in ((0, 50), (1, 44), (6840, 6860), (163 * 42 - 1, 163 * 42 + 1), (b - 30, b)):
            sub = slice(lo * 3, hi * 3)
            sub_kw = {k: None if a is None else a[sub] for k, a in kw.items()}
            sv, sd, sj = eng.kg_qbatch(c["xq"][sub], q, nf, Eb, **sub_kw)
            assert np.array_equal(sv, v[lo:hi]) and np.array_equal(sj, jit[lo:hi]), (lo, hi)
            assert np.array_equal(sd, d[sub]), (lo, hi)
        dev = {k: None if a is None else torch.from_numpy(a[:300]).cuda() for k, a in kw.items()}
        xd = torch.from_numpy(c["xq"][:300]).cuda()
        vd = torch.empty(100, dtype=torch.float64, device="cuda")
        dd = torch.empty(300, 32, dtype=torch.float64, device="cuda")
        eng.kg_qbatch(xd, q, nf, torch.from_numpy(Eb).cuda(), out_values=vd, out_d_xq=dd, **dev)
        assert np.array_equal(vd.cpu().numpy(), v[:100]) and np.array_equal(dd.cpu().numpy(), d[:300])
    finally:
        eng.close()


def test_zero_base_samples_give_the_fantasy_means():
    """e = 0: every term is the fantasy row's posterior mean, Sigma_bar and the actual rows' mu_bar vanish, so d_xq is
    exactly 0 on the actual rows and sigma/F times predict_grad's d_mean on the fantasy rows."""
    p = make_problem(300, 3, 2, n_noise=2, n_mean=2, seed=40)
    q, nf, b = 3, 5, 20
    c = make_candidates(p, b * (q + nf), seed=41)
    kw = _kw(c)
    eng = _engine(p)
    try:
        eng.factorize(make_hyper(p, seed=14, noise=1e-2))
        mean, _ = eng.posterior_qbatch(c["xq"], q + nf, include_noise=True, **kw)
        mu, _, d_mean, _ = eng.predict_grad(c["xq"], **kw)
        for maximize in (True, False):
            sgn = 1.0 if maximize else -1.0
            v, d, _ = eng.kg_qbatch(c["xq"], q, nf, np.zeros((nf, q)), maximize=maximize, **kw)
            want_v = np.array([sgn * sum(float(x) for x in row) * (1.0 / nf) for row in mean[:, q:]])
            np.testing.assert_allclose(v, want_v, rtol=1e-15, atol=0)
            d = d.reshape(b, q + nf, -1)
            assert np.array_equal(d[:, :q], np.zeros_like(d[:, :q]))
            want = sgn / nf * d_mean.reshape(b, q + nf, -1)[:, q:]
            err = float(np.abs(d[:, q:] - want).max()) / float(np.abs(want).max())
            print("zero samples: d_xq of the fantasy rows vs predict_grad %.2e" % err)
            assert err <= GRAD_TOL
    finally:
        eng.close()


def test_gradient_matches_central_differences():
    p = make_problem(200, 3, 2, dz=2, n_combo=3, n_noise=2, n_mean=2, seed=21)
    h = make_hyper(p, seed=11, noise=1e-2)
    q, nf, b = 2, 3, 3
    c = make_candidates(p, b * (q + nf), seed=22)
    kw = _kw(c)
    Eb = _base(nf, q, seed=1)
    eng = _engine(p)
    try:
        eng.factorize(h)
        _, d, _ = eng.kg_qbatch(c["xq"], q, nf, Eb, **kw)

        def f(x):
            return float(eng.kg_qbatch(x, q, nf, Eb, want_grad=False, **kw)[0].sum())

        eps = 1e-6
        fd = np.zeros_like(d)
        for i in range(b * (q + nf)):
            for k in range(p["dq"]):
                xp, xm = c["xq"].copy(), c["xq"].copy()
                xp[i, k] += eps
                xm[i, k] -= eps
                fd[i, k] = (f(xp) - f(xm)) / (2 * eps)
        print("d_xq vs central differences %.2e" % float(np.max(np.abs(d - fd))))
        np.testing.assert_allclose(d, fd, rtol=1e-5, atol=1e-6)
    finally:
        eng.close()


def test_jitter_only_where_the_block_needs_it():
    """t-batch 1's actual rows repeat one point far from every training point, in a noise group without noise: its A
    is exactly the all-ones matrix (sigma_f^2 = 1), whose second pivot is exactly 0, and 1e-8 I makes it decisively
    positive definite, so the ladder gives 1e-8 whichever Cholesky runs it.  The other t-batches take no jitter."""
    p = make_problem(200, 3, 0, n_noise=2, seed=32)
    p["noise_idx"] = np.zeros(200, dtype=np.int32)
    q, nf, b = 6, 3, 4
    c = make_candidates(p, b * (q + nf), seed=33)
    c["noise_idx"] = np.zeros(b * (q + nf), dtype=np.int32)
    r = q + nf
    c["xq"][r:r + q] = 1e3
    c["xq"][r + q:2 * r] = 1e3 + 0.3 * np.random.default_rng(2).standard_normal((nf, 3))
    c["noise_idx"][r:r + q] = 1
    h = make_hyper(p, seed=13, noise=1e-4)
    h["sigma_f2"] = 1.0
    h["noise"] = np.array([1e-4, 0.0])
    E = _base(nf, q)
    eng = _engine(p)
    try:
        eng.factorize(h)
        mean, cov = eng.posterior_qbatch(c["xq"], r, include_noise=True, **_kw(c))
        v, d, jit = eng.kg_qbatch(c["xq"], q, nf, E, **_kw(c))
    finally:
        eng.close()
    assert np.array_equal(cov[1, :q, :q], np.ones((q, q)))
    want = ladder_jitter(torch.from_numpy(cov[:, :q, :q])).numpy()
    cond = [float(np.linalg.cond(cov[t, :q, :q])) for t in (0, 2, 3)]
    vt, _, _, _ = kg_block(mean, cov, q, E, True, jit)
    print("jitter per t-batch", jit, "ladder", want, "cond of the others", cond, "value vs torch %.2e"
          % float(np.max(np.abs(v - vt))))
    assert max(cond) < 1e6
    assert np.array_equal(jit, want) and np.array_equal(jit, [0.0, 1e-8, 0.0, 0.0])
    assert float(np.max(np.abs(v - vt))) <= VAL_TOL_ENGINE
    assert np.all(np.isfinite(v)) and np.all(np.isfinite(d))


def test_argument_and_status_codes():
    from gpplus_b200 import _engine as E
    p = make_problem(100, 2, 0, seed=24)
    eng = _engine(p)
    try:
        eng.factorize(make_hyper(p, seed=1))
        x = np.ascontiguousarray(make_candidates(p, 129 * 2, seed=25)["xq"])
        Eb = _base(4, 4)
        vals = np.empty(2)
        lib, h = eng._lib, eng._h
        for b, q, nf, base, out, match in ((2, 0, 4, Eb, vals, b"n_fantasies"), (2, 4, 0, Eb, vals, b"n_fantasies"),
                                           (2, 64, 65, Eb, vals, b"GPP_MAX_QBATCH"), (-1, 4, 4, Eb, vals, b"b must"),
                                           (2, 4, 4, None, vals, b"missing"), (2, 4, 4, Eb, None, b"missing")):
            rc = lib.gpp_kg_qbatch(h, b, q, nf, E._ptr(x), None, None, None, 1, E._ptr(base), E._ptr(out), None, None)
            assert rc == E.GPP_ERR_ARG and match in lib.gpp_last_error(), (b, q, nf)
        with pytest.raises(ValueError, match="base_samples must have shape"):
            eng.kg_qbatch(x[:16], 4, 4, _base(4, 3))
        with pytest.raises(ValueError, match="n_fantasies"):
            eng.kg_qbatch(x[:16], 4, 0, Eb)
        v, d, jit = eng.kg_qbatch(x[:0], 4, 4, Eb)
        assert v.shape == (0,) and jit.shape == (0,)
        xn = x[:16].copy()
        xn[9, 1] = np.nan
        with pytest.raises(Exception, match="NaN"):
            eng.kg_qbatch(xn, 4, 4, Eb)
    finally:
        eng.close()
    # a t-batch whose actual rows' block fails every rung: two identical points far from the training set in a noise
    # group of -1e-5 make A = ones - 1e-5 I (sigma_f^2 = 1), indefinite at every rung of the ladder
    p = make_problem(100, 2, 0, n_noise=2, seed=26)
    p["noise_idx"] = np.zeros(100, dtype=np.int32)
    h = make_hyper(p, seed=2)
    h["sigma_f2"] = 1.0
    h["noise"] = np.array([1e-3, -1e-5])
    c = make_candidates(p, 2 * 4, seed=27)
    c["xq"][:2] = 1e3
    c["noise_idx"] = np.array([1, 1, 0, 0, 0, 0, 0, 0], dtype=np.int32)
    eng = _engine(p)
    try:
        eng.factorize(h)
        with pytest.raises(Exception, match="not positive definite"):
            eng.kg_qbatch(c["xq"], 2, 2, _base(2, 2), noise_idx=c["noise_idx"])
    finally:
        eng.close()


def _mf_model():
    """Two sources of one 2-D function (source 1 a cheap, biased copy), source column last."""
    from gpplus_b200.models import GP_Plus
    rng = np.random.default_rng(50)
    n0, n1 = 12, 30
    X = np.vstack([np.hstack([rng.uniform(-2, 2, (n0, 2)), np.zeros((n0, 1))]),
                   np.hstack([rng.uniform(-2, 2, (n1, 2)), np.ones((n1, 1))])])
    f = -(X[:, 0] - 0.5) ** 2 - 0.5 * (X[:, 1] + 0.3) ** 2 + 0.3 * np.sin(3 * X[:, 0])
    y = f + (X[:, 2] == 1) * (0.2 * X[:, 0] - 0.1) + 0.01 * rng.standard_normal(n0 + n1)
    m = GP_Plus(torch.tensor(X), torch.tensor(y), qual_dict={2: 2}, multiple_noise=True, dtype=torch.float64)
    return m


def test_cost_aware_multi_fidelity_kg_end_to_end():
    from gpplus_b200.bayesian_optimizations import optimize_knowledge_gradient, optimize_posterior_mean
    m = _mf_model()
    bounds = np.array([[-2.0, -2.0], [2.0, 2.0]])
    target, cost = 0, {0: 10.0, 1: 1.0}
    x_best, cur = optimize_posterior_mean(m, bounds, fixed_columns={2: target}, num_restarts=4, raw_samples=64,
                                          options={"maxiter": 30}, seed=3)
    with torch.no_grad():
        assert cur == pytest.approx(float(m.predict(x_best[None], return_std=False)[0]), rel=1e-12)
    q, nf = 2, 16
    seen = []
    orig = m.knowledge_gradient

    def spy(Xc, n, **kw):
        v = orig(Xc, n, **kw)
        seen.append((Xc.detach().clone(), v.detach().clone()))
        return v

    m.knowledge_gradient = spy
    for source in (0, 1):
        args = dict(num_fantasies=nf, fixed_columns={2: source}, fantasy_fixed_columns={2: target}, num_restarts=4,
                    raw_samples=64, options={"maxiter": 30}, seed=5, current_value=cur, cost_by_source=cost)
        X, v = optimize_knowledge_gradient(m, bounds, q, **args)
        assert X.shape == (q, 3) and bool((X[:, 2] == source).all()) and bool((X[:, :2].abs() <= 2.0).all())
        # the screening of the optimiser, repeated: its best value is a floor for the result
        from gpplus_b200.models.gpregression import sobol_normal_samples
        E = sobol_normal_samples(nf, q, 5)
        raw = torch.quasirandom.SobolEngine(dimension=(q + nf) * 2, scramble=True, seed=5).draw(64, dtype=torch.float64)
        Xr = torch.zeros(64, q + nf, 3, dtype=torch.float64)
        Xr[:, :, :2] = -2.0 + 4.0 * raw.reshape(64, q + nf, 2)
        Xr[:, :q, 2] = source
        Xr[:, q:, 2] = target
        with torch.no_grad():
            v_raw = m.knowledge_gradient(Xr, nf, base_samples=E, current_value=cur, cost_by_source=cost)
        print("source %d: optimised cost-aware KG %.6g, best screened %.6g" % (source, v, float(v_raw.max())))
        assert v >= float(v_raw.max())
        assert np.isfinite(v)
        # the value belongs to an evaluated t-batch with these actual rows, and that t-batch alone re-evaluates to it
        hits = [(Xc[i], vc[i]) for Xc, vc in seen for i in range(Xc.shape[0])
                if torch.equal(Xc[i, :q], X) and float(vc[i]) == v]
        assert hits
        with torch.no_grad():
            again = orig(hits[-1][0][None], nf, base_samples=E, current_value=cur, cost_by_source=cost)
        assert float(again[0]) == v
    m.release_engine()
