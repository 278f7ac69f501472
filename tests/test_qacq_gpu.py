"""gpp_acq_qbatch on the B200: Monte-Carlo qEI / qNEI / qUCB values and input gradients against torch on the engine's
own t-batch posteriors and against the dense CPU reference (tests/qacq_reference.py), bitwise identities (repeated,
values-only, sub-ranges across chunk boundaries, device-resident), central differences, the q = 1 limits, the
per-t-batch jitter, argument checks, and GPR.acquisition_qbatch / optimize_acquisition_qbatch end to end."""
import math

import numpy as np
import pytest
import torch

from problems import engine_kwargs, make_candidates, make_hyper, make_problem
from qacq_reference import KINDS, acq_qbatch as reference_acq, ladder_jitter, mc_utility

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


def _kw(c, include_noise):
    return dict(level_idx=c["level_idx"], noise_idx=c["noise_idx"], mean_idx=c["mean_idx"], include_noise=include_noise)


def _base(S, q_tot, seed=0):
    from gpplus_b200.models.gpregression import sobol_normal_samples
    return np.ascontiguousarray(sobol_normal_samples(S, q_tot, seed).numpy())


def _params(kind, q_tot, mean):
    n_base = max(1, q_tot // 4) if kind == "NEI" else 0
    return dict(kind=KINDS[kind], best_f=float(np.quantile(mean, 0.7)), beta=0.8, n_baseline=n_base)


def _check(p, h, c, q_tot, kind, include_noise=False, fp64=None, S=64, maximize=True):
    b = c["m"] // q_tot
    kw = _kw(c, include_noise)
    E = _base(S, q_tot, seed=q_tot)
    eng = _engine(p, fp64)
    try:
        eng.factorize(h)
        mu0, var0 = eng.predict(c["xq"], min_var=-np.inf, **kw)
        alpha0, stats0 = eng.fetch("alpha"), eng.stats()
        mean, cov = eng.posterior_qbatch(c["xq"], q_tot, **kw)
        a = _params(kind, q_tot, mean)
        args = dict(best_f=a["best_f"], beta=a["beta"], n_baseline=a["n_baseline"], maximize=maximize, **kw)
        v, d, jit = eng.acquisition_qbatch(c["xq"], q_tot, a["kind"], E, **args)
        v1, d1, jit1 = eng.acquisition_qbatch(c["xq"], q_tot, a["kind"], E, **args)
        v0, none, jit0 = eng.acquisition_qbatch(c["xq"], q_tot, a["kind"], E, want_grad=False, **args)
        vt, gm, gc, _ = mc_utility(mean, cov, E, a["kind"], a["best_f"], a["beta"], a["n_baseline"], maximize, jit)
        d_eng = eng.posterior_qbatch_grad(c["xq"], q_tot, gm, gc, **kw)
        mu1, var1 = eng.predict(c["xq"], min_var=-np.inf, **kw)
        assert np.array_equal(eng.fetch("alpha"), alpha0) and np.array_equal(mu1, mu0) and np.array_equal(var1, var0)
        assert eng.stats() == stats0
    finally:
        eng.close()
    assert v.shape == (b,) and d.shape == (b * q_tot, p["dq"]) and jit.shape == (b,) and none is None
    assert np.all(np.isfinite(v)) and np.all(np.isfinite(d))
    assert np.array_equal(v, v1) and np.array_equal(d, d1) and np.array_equal(jit, jit1), "repeated calls differ"
    assert np.array_equal(v0, v) and np.array_equal(jit0, jit), "values-only differs from the gradient call"
    cond = float(np.max(np.linalg.cond(cov + jit[:, None, None] * np.eye(q_tot))))
    verr = float(np.max(np.abs(v - vt)))
    scale = max(1.0, float(np.max(np.abs(d_eng), initial=0.0)))
    derr = float(np.max(np.abs(d - d_eng), initial=0.0)) / scale
    print("%s q_tot=%d b=%d cond %.1e jitter %.0e: engine blocks value %.2e d_xq %.2e"
          % (kind, q_tot, b, cond, float(jit.max()), verr, derr))
    assert cond < 1e6, cond
    assert verr <= VAL_TOL_ENGINE, verr
    assert derr <= GRAD_TOL, derr
    rv, rd, _ = reference_acq(p, h, c, q_tot, a["kind"], E, a["best_f"], a["beta"], a["n_baseline"], maximize,
                              include_noise, jit)
    rverr = float(np.max(np.abs(v - rv)))
    rderr = float(np.max(np.abs(d - rd), initial=0.0)) / max(1.0, float(np.max(np.abs(rd), initial=0.0)))
    print("   dense reference: value %.2e d_xq %.2e" % (rverr, rderr))
    assert rverr <= VAL_TOL_DENSE, rverr
    assert rderr <= GRAD_TOL, rderr
    return v, d, jit


@pytest.mark.parametrize("kind", ["EI", "NEI", "UCB"])
@pytest.mark.parametrize("kernel", [0, 1, 2])
@pytest.mark.parametrize("q_tot", [1, 3, 8, 64, 128])
def test_kinds_kernels_and_batch_sizes(kind, kernel, q_tot):
    if kind == "NEI" and q_tot == 1:
        pytest.skip("qNEI needs at least one candidate and one baseline row")
    p = make_problem(300, 4, kernel, seed=kernel + 1)
    b = max(2, 384 // q_tot)
    _check(p, make_hyper(p, seed=3, noise=1e-2), make_candidates(p, b * q_tot, seed=q_tot), q_tot, kind,
           include_noise=True, maximize=kernel != 1)


@pytest.mark.parametrize("n_pass", [1, 3])
def test_latent_map_and_ensemble(n_pass):
    p = make_problem(260, 3, 2, dz=2, n_combo=6, n_pass=n_pass, seed=11)
    _check(p, make_hyper(p, seed=4, noise=1e-2), make_candidates(p, 40 * 5, seed=6), 5, "NEI", include_noise=True)


@pytest.mark.parametrize("include_noise", [False, True])
def test_noise_groups_and_means(include_noise):
    p = make_problem(300, 5, 1, dz=2, n_combo=4, n_noise=3, n_mean=3, zero_mean_group=True, seed=12)
    _check(p, make_hyper(p, seed=5, noise=1e-2), make_candidates(p, 37 * 7, seed=7), 7, "EI",
           include_noise=include_noise)


@pytest.mark.parametrize("dq", [0, 32])
def test_input_widths(dq):
    if dq == 0:
        p = make_problem(200, 0, 0, dz=2, n_combo=5, seed=14)
        h = make_hyper(p, seed=7, noise=1e-2)
    else:
        p = make_problem(400, 32, 2, seed=13)
        h = make_hyper(p, seed=6, noise=1e-2, w_scale=0.02)
    _check(p, h, make_candidates(p, 30 * 6, seed=8), 6, "UCB", include_noise=True)


@pytest.mark.parametrize("fp64", ["dmma", "int8"])
def test_int8_sliced_factor(fp64):
    from gpplus_b200 import _engine as E
    p = make_problem(3200, 4, 2, seed=15)
    _check(p, make_hyper(p, seed=8, noise=1e-2), make_candidates(p, 60 * 8, seed=10), 8, "EI", include_noise=True,
           fp64=E.FP64_DMMA if fp64 == "dmma" else E.FP64_INT8)


def test_other_batches_and_chunk_split_do_not_matter():
    """N = 3200, dq = 32, q_tot = 3: chunks of 163 tiles of 42 t-batches, so 13 709 t-batches take three chunks.  Any
    run of t-batches called alone gives bitwise the full call's values, jitters and gradients, and so do
    device-resident inputs and outputs."""
    from gpplus_b200 import _engine as E
    p = make_problem(3200, 32, 2, seed=18)
    h = make_hyper(p, seed=10, noise=1e-3, w_scale=0.02)
    q, b = 3, 163 * 42 * 2 + 17
    c = make_candidates(p, b * q, seed=19)
    Eb = _base(32, q, seed=5)
    args = dict(best_f=0.2, n_baseline=1)
    eng = _engine(p)
    try:
        eng.factorize(h)
        v, d, jit = eng.acquisition_qbatch(c["xq"], q, E.QACQ_NEI, Eb, **args)
        for lo, hi in ((0, 50), (1, 44), (6840, 6860), (163 * 42 - 1, 163 * 42 + 1), (b - 30, b)):
            sub = slice(lo * q, hi * q)
            sv, sd, sj = eng.acquisition_qbatch(c["xq"][sub], q, E.QACQ_NEI, Eb, **args)
            assert np.array_equal(sv, v[lo:hi]) and np.array_equal(sj, jit[lo:hi]), (lo, hi)
            assert np.array_equal(sd, d[sub]), (lo, hi)
        xd = torch.from_numpy(c["xq"][:300]).cuda()
        vd = torch.empty(100, dtype=torch.float64, device="cuda")
        dd = torch.empty(300, 32, dtype=torch.float64, device="cuda")
        eng.acquisition_qbatch(xd, q, E.QACQ_NEI, torch.from_numpy(Eb).cuda(), out_values=vd, out_d_xq=dd, **args)
        assert np.array_equal(vd.cpu().numpy(), v[:100]) and np.array_equal(dd.cpu().numpy(), d[:300])
    finally:
        eng.close()


def test_gradient_matches_central_differences():
    p = make_problem(200, 3, 2, dz=2, n_combo=3, n_noise=2, n_mean=2, seed=21)
    h = make_hyper(p, seed=11, noise=1e-2)
    q, b = 4, 3
    c = make_candidates(p, b * q, seed=22)
    Eb = _base(64, q, seed=1)
    eng = _engine(p)
    try:
        eng.factorize(h)
        for kind, args in ((KINDS["EI"], dict(best_f=0.0)), (KINDS["NEI"], dict(n_baseline=1)),
                           (KINDS["UCB"], dict(beta=1.5))):
            _, d, _ = eng.acquisition_qbatch(c["xq"], q, kind, Eb, **args, **_kw(c, True))

            def f(x):
                return float(eng.acquisition_qbatch(x, q, kind, Eb, want_grad=False, **args, **_kw(c, True))[0].sum())

            eps = 1e-6
            fd = np.zeros_like(d)
            for i in range(b * q):
                for k in range(p["dq"]):
                    xp, xm = c["xq"].copy(), c["xq"].copy()
                    xp[i, k] += eps
                    xm[i, k] -= eps
                    fd[i, k] = (f(xp) - f(xm)) / (2 * eps)
            print("kind %d: d_xq vs central differences %.2e" % (kind, float(np.max(np.abs(d - fd)))))
            np.testing.assert_allclose(d, fd, rtol=1e-5, atol=1e-6)
    finally:
        eng.close()


def test_single_point_limits():
    """q_tot = 1 with 2^14 Sobol samples: qEI -> sigma (phi(u) + u Phi(u)), qUCB -> mu + sqrt(beta) sigma."""
    from gpplus_b200 import _engine as E
    p = make_problem(300, 3, 2, seed=30)
    c = make_candidates(p, 20, seed=31)
    Eb = _base(1 << 14, 1, seed=2)
    eng = _engine(p)
    try:
        eng.factorize(make_hyper(p, seed=12, noise=1e-2))
        mu, var = eng.predict(c["xq"], min_var=-np.inf)
        best_f, beta = float(np.median(mu)), 2.0
        vei, _, _ = eng.acquisition_qbatch(c["xq"], 1, E.QACQ_EI, Eb, best_f=best_f, want_grad=False)
        vucb, _, _ = eng.acquisition_qbatch(c["xq"], 1, E.QACQ_UCB, Eb, beta=beta, want_grad=False)
    finally:
        eng.close()
    sd = np.sqrt(var)
    u = (mu - best_f) / sd
    phi = np.exp(-0.5 * u * u) / math.sqrt(2 * math.pi)
    Phi = 0.5 * (1 + np.array([math.erf(x / math.sqrt(2)) for x in u]))
    ei = sd * (phi + u * Phi)
    ucb = mu + math.sqrt(beta) * sd
    # relative accuracy of the quadrature holds where the improvement is not a far tail event
    body = np.abs(u) <= 1.5
    assert np.count_nonzero(body) >= 5
    print("q=1 limits: qEI %.2e (%d points with |u| <= 1.5), qUCB %.2e (relative)"
          % (float(np.max(np.abs(vei - ei)[body] / ei[body])), int(np.count_nonzero(body)),
             float(np.max(np.abs(vucb - ucb) / np.abs(ucb)))))
    np.testing.assert_allclose(vei[body], ei[body], rtol=2e-3)
    np.testing.assert_allclose(vucb, ucb, rtol=2e-3)


def test_jitter_only_where_the_block_needs_it():
    """t-batch 1 repeats one point far from every training point: its K* row is below the smallest double, so U = 0
    and, with sigma_f^2 = 1, its block is exactly the all-ones matrix.  The second pivot of that block is exactly 0 in
    any arithmetic (rung 0 fails) and 1e-8 I makes it decisively positive definite, so the ladder gives 1e-8 whichever
    Cholesky runs it.  The other t-batches are well conditioned and take no jitter."""
    from gpplus_b200 import _engine as E
    p = make_problem(200, 3, 0, seed=32)
    q, b = 8, 4
    c = make_candidates(p, b * q, seed=33)
    c["xq"][q:2 * q] = 1e3
    h = make_hyper(p, seed=13, noise=1e-4)
    h["sigma_f2"] = 1.0
    Eb = _base(32, q)
    eng = _engine(p)
    try:
        eng.factorize(h)
        _, cov = eng.posterior_qbatch(c["xq"], q)
        v, d, jit = eng.acquisition_qbatch(c["xq"], q, E.QACQ_EI, Eb, best_f=0.0)
    finally:
        eng.close()
    assert np.array_equal(cov[1], np.ones((q, q)))
    want = ladder_jitter(torch.from_numpy(cov)).numpy()
    cond = [float(np.linalg.cond(cov[t])) for t in (0, 2, 3)]
    print("jitter per t-batch", jit, "ladder", want, "cond of the others", cond)
    assert max(cond) < 1e6
    assert np.array_equal(jit, want) and np.array_equal(jit, [0.0, 1e-8, 0.0, 0.0])
    assert np.all(np.isfinite(v)) and np.all(np.isfinite(d))


def test_argument_checks():
    import ctypes as C
    from gpplus_b200 import _engine as E
    p = make_problem(100, 2, 0, seed=24)
    eng = _engine(p)
    try:
        eng.factorize(make_hyper(p, seed=1))
        x = make_candidates(p, 129 * 2, seed=25)["xq"]
        Eb = _base(8, 4)
        for kind, nb, match in ((3, 0, "kind"), (E.QACQ_NEI, 0, "n_baseline"), (E.QACQ_NEI, 4, "n_baseline"),
                                (E.QACQ_EI, 1, "n_baseline"), (E.QACQ_UCB, 2, "n_baseline")):
            with pytest.raises(ValueError, match=match):
                eng.acquisition_qbatch(x[:8], 4, kind, Eb, n_baseline=nb)
        with pytest.raises(ValueError, match="GPP_MAX_QBATCH"):
            eng.acquisition_qbatch(x, 129, E.QACQ_EI, _base(8, 129))
        with pytest.raises(ValueError, match="GPP_MAX_MC_SAMPLES"):
            eng.acquisition_qbatch(x[:4], 1, E.QACQ_EI, np.zeros((E.MAX_MC_SAMPLES + 1, 1)))
        with pytest.raises(ValueError, match="GPP_MAX_MC_SAMPLES"):
            eng.acquisition_qbatch(x[:4], 1, E.QACQ_EI, np.zeros((0, 1)))
        with pytest.raises(ValueError, match="beta"):
            eng.acquisition_qbatch(x[:8], 4, E.QACQ_UCB, Eb, beta=-1.0)
        xq = np.ascontiguousarray(x[:8])
        vals = np.empty(2)
        for base, out in ((None, vals), (Eb, None)):
            rc = eng._lib.gpp_acq_qbatch(eng._h, 2, 4, E._ptr(xq), None, None, None, 0, E.QACQ_EI, 0, 0.0, 0.0, 1, 8,
                                         E._ptr(base), E._ptr(out), None, None)
            assert rc == E.GPP_ERR_ARG and b"missing" in eng._lib.gpp_last_error()
        v, d, jit = eng.acquisition_qbatch(x[:0], 4, E.QACQ_EI, Eb)
        assert v.shape == (0,) and jit.shape == (0,)
    finally:
        eng.close()


def _qei_model():
    from gpplus_b200.models import GP_Plus
    rng = np.random.default_rng(26)
    X = rng.uniform(-2, 2, (80, 3))
    y = np.sin(X[:, 0]) + 0.5 * np.cos(1.5 * X[:, 1]) + 0.2 * X[:, 2] + 0.02 * rng.standard_normal(80)
    m = GP_Plus(torch.tensor(X), torch.tensor(y), dtype=torch.float64, quant_correlation_class="Matern52Kernel")
    with torch.no_grad():
        m.covar_module.raw_outputscale.fill_(0.5)
    return m, y, rng


def test_model_matches_torch_qei_and_the_optimizer_improves_on_screening():
    """GPR.acquisition_qbatch against the torch qEI of the q-batch posterior test with the same base samples expanded
    over the t-batches, then optimize_acquisition_qbatch for q = 4."""
    from gpplus_b200.bayesian_optimizations import optimize_acquisition_qbatch
    m, y, rng = _qei_model()
    b, q, S = 4, 3, 256
    E1 = torch.randn(S, q, generator=torch.Generator().manual_seed(3), dtype=torch.float64)
    best_sc = float(np.quantile((y - float(m.y_min)) / float(m.y_std), 0.75))
    best = float(m.y_min) + float(m.y_std) * best_sc
    x0 = torch.tensor(rng.uniform(-2, 2, (b, q, 3)))

    x = x0.clone().requires_grad_(True)
    post = m.posterior(x, observation_noise=False)
    f = post.rsample(torch.Size([S]), base_samples=E1[:, None, :].expand(S, b, q))
    ref = float(m.y_std) * (f - best_sc).clamp_min(0).max(-1).values.mean(0)
    g_ref, = torch.autograd.grad(ref.sum(), x)
    xe = x0.clone().requires_grad_(True)
    val = m.acquisition_qbatch(xe, "qEI", best_f=best, base_samples=E1)
    g, = torch.autograd.grad(val.sum(), xe)
    print("model qEI vs torch: values %.2e, gradients %.2e" % (
        float(((val - ref).abs() / ref.abs().clamp_min(1e-300)).max()),
        float((g - g_ref).abs().max() / g_ref.abs().max())))
    np.testing.assert_allclose(val.detach().numpy(), ref.detach().numpy(), rtol=1e-9)
    assert float((g - g_ref).abs().max()) <= 1e-7 * float(g_ref.abs().max())

    bounds = np.array([[-2.0] * 3, [2.0] * 3])
    Xopt, vopt = optimize_acquisition_qbatch(m, bounds, 4, "qEI", num_restarts=4, raw_samples=64,
                                             options={"maxiter": 40}, seed=7, best_f=best, num_samples=256)
    from gpplus_b200.models.gpregression import sobol_normal_samples
    raw = torch.quasirandom.SobolEngine(dimension=12, scramble=True, seed=7).draw(64, dtype=torch.float64)
    with torch.no_grad():
        v_raw = m.acquisition_qbatch(-2.0 + 4.0 * raw.reshape(64, 4, 3), "qEI", best_f=best,
                                     base_samples=sobol_normal_samples(256, 4, 7))
    print("optimised qEI %.6f, best raw %.6f" % (vopt, float(v_raw.max())))
    assert Xopt.shape == (4, 3) and bool((Xopt.abs() <= 2.0).all())
    assert vopt > float(v_raw.max())
    m.release_engine()
