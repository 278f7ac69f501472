"""gpp_posterior_qbatch / gpp_posterior_qbatch_grad on the B200: the t-batch joint posteriors and their input
gradients against the dense CPU reference (tests/qbatch_posterior_reference.py), their exact relations to gpp_predict
and gpp_predict_joint, independence of the other t-batches and of the chunk split, the untouched handle state, and a
Monte-Carlo qEI optimised with L-BFGS-B through GPR.posterior on a [b, q, d] batch."""
import numpy as np
import pytest
import torch

from problems import engine_kwargs, make_candidates, make_hyper, make_problem

pytestmark = pytest.mark.gpu

# |Sigma_engine - Sigma_ref| per entry relative to sigma_f^2: the bound of the gpp_predict_joint tests, whose U this is
COV_TOL = 1e-9
# |d_xq - d_ref| relative to the largest |d_ref| of the case (room for the INT8-sliced factor, which feeds U and V)
GRAD_TOL = 1e-7


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


def _rows(c, lo, hi):
    out = {k: (v[lo:hi] if isinstance(v, np.ndarray) else v) for k, v in c.items()}
    out["m"] = hi - lo
    return out


def _upstream(b, q, seed):
    rng = np.random.default_rng(seed)
    return rng.standard_normal((b, q)), rng.standard_normal((b, q, q))


def _check(p, h, c, q, include_noise=False, fp64=None):
    from qbatch_posterior_reference import posterior_qbatch as reference
    b = c["m"] // q
    gm, gc = _upstream(b, q, seed=q)
    kw = _kw(c, include_noise)
    eng = _engine(p, fp64)
    try:
        eng.factorize(h)
        mu0, var0 = eng.predict(c["xq"], min_var=-np.inf, **kw)
        alpha0 = eng.fetch("alpha")
        mean, cov = eng.posterior_qbatch(c["xq"], q, **kw)
        d = eng.posterior_qbatch_grad(c["xq"], q, gm, gc, **kw)
        again = eng.posterior_qbatch(c["xq"], q, **kw)
        d_again = eng.posterior_qbatch_grad(c["xq"], q, gm, gc, **kw)
        mu1, var1 = eng.predict(c["xq"], min_var=-np.inf, **kw)
        assert np.array_equal(eng.fetch("alpha"), alpha0) and np.array_equal(mu1, mu0) and np.array_equal(var1, var0)
        blocks = sorted({0, b // 2, b - 1})
        joint = {t: eng.predict_joint(c["xq"][t * q:(t + 1) * q], **_kw(_rows(c, t * q, (t + 1) * q), include_noise))[1]
                 for t in blocks}
    finally:
        eng.close()
    sf2 = h["sigma_f2"]
    assert mean.shape == (b, q) and cov.shape == (b, q, q) and d.shape == (b * q, p["dq"])
    assert np.all(np.isfinite(cov)) and np.all(np.isfinite(d))
    assert np.array_equal(mean.reshape(-1), mu0), "mean is not bitwise gpp_predict's"
    assert np.array_equal(np.diagonal(cov, axis1=1, axis2=2).reshape(-1), var0), "diagonal is not gpp_predict's"
    assert np.array_equal(cov, cov.transpose(0, 2, 1)), "a block is not exactly symmetric"
    assert np.array_equal(mean, again[0]) and np.array_equal(cov, again[1]) and np.array_equal(d, d_again), \
        "repeated calls differ"
    for t in blocks:
        assert np.max(np.abs(cov[t] - joint[t])) <= COV_TOL * sf2, "block %d differs from predict_joint" % t
    rmean, rcov, rd = reference(p, h, c, q, include_noise, gm, gc)
    cerr = float(np.max(np.abs(cov - rcov))) / sf2
    derr = float(np.max(np.abs(d - rd), initial=0.0)) / max(1.0, float(np.max(np.abs(rd), initial=0.0)))
    print("q=%d b=%d cov err %.2e (sigma_f^2 units), d_xq err %.2e (relative)" % (q, b, cerr, derr))
    assert cerr <= COV_TOL, cerr
    assert derr <= GRAD_TOL, derr
    assert np.max(np.abs(mean - rmean)) <= 1e-8
    return mean, cov, d


@pytest.mark.parametrize("kernel", [0, 1, 2])
@pytest.mark.parametrize("q", [1, 3, 8, 64, 128])
def test_kernels_and_batch_sizes(kernel, q):
    p = make_problem(300, 4, kernel, seed=kernel + 1)
    b = max(3, 700 // q)
    _check(p, make_hyper(p, seed=3), make_candidates(p, b * q, seed=q), q)


@pytest.mark.parametrize("n_pass", [1, 3])
def test_latent_map_and_ensemble(n_pass):
    p = make_problem(260, 3, 2, dz=2, n_combo=6, n_pass=n_pass, seed=11)
    _check(p, make_hyper(p, seed=4), make_candidates(p, 40 * 5, seed=6), 5)


@pytest.mark.parametrize("include_noise", [False, True])
def test_noise_groups_and_means(include_noise):
    p = make_problem(300, 5, 1, dz=2, n_combo=4, n_noise=3, n_mean=3, zero_mean_group=True, seed=12)
    _check(p, make_hyper(p, seed=5, noise=1e-2), make_candidates(p, 37 * 7, seed=7), 7, include_noise=include_noise)


@pytest.mark.parametrize("dq", [0, 32])
def test_input_widths(dq):
    if dq == 0:
        p = make_problem(200, 0, 0, dz=2, n_combo=5, seed=14)
        h = make_hyper(p, seed=7)
    else:
        p = make_problem(400, 32, 2, seed=13)
        h = make_hyper(p, seed=6, w_scale=0.02)
    _check(p, h, make_candidates(p, 30 * 6, seed=8), 6)


@pytest.mark.parametrize("fp64", ["dmma", "int8"])
def test_int8_sliced_factor(fp64):
    from gpplus_b200 import _engine as E
    p = make_problem(3200, 4, 2, seed=15)
    _check(p, make_hyper(p, seed=8, noise=1e-3), make_candidates(p, 60 * 8, seed=10), 8,
           fp64=E.FP64_DMMA if fp64 == "dmma" else E.FP64_INT8)


def test_single_point_batches_are_gpp_predict():
    p = make_problem(500, 3, 1, n_noise=2, seed=16)
    c = make_candidates(p, 1000, seed=17)
    c["xq"][:5] = p["xq"][:5]  # candidates on training points: variances near the noise level
    eng = _engine(p)
    try:
        eng.factorize(make_hyper(p, seed=9, noise=1e-4))
        for noise in (False, True):
            mu0, var0 = eng.predict(c["xq"], min_var=-np.inf, **_kw(c, noise))
            mean, cov = eng.posterior_qbatch(c["xq"], 1, **_kw(c, noise))
            assert np.array_equal(mean[:, 0], mu0) and np.array_equal(cov[:, 0, 0], var0)
    finally:
        eng.close()


def test_other_batches_and_chunk_split_do_not_matter():
    """N = 3200, dq = 32: the t-batch path runs chunks of 20 864 rows (163 tiles of 42 t-batches of q = 3), so
    13 709 t-batches take three chunks.  Any run of t-batches called alone, at another slot of its tiles or across a
    chunk boundary of the full call, gives bitwise the same means, blocks and gradients."""
    p = make_problem(3200, 32, 2, seed=18)
    h = make_hyper(p, seed=10, noise=1e-3, w_scale=0.02)
    q, b = 3, 163 * 42 * 2 + 17
    c = make_candidates(p, b * q, seed=19)
    gm, gc = _upstream(b, q, seed=20)
    eng = _engine(p)
    try:
        eng.factorize(h)
        mean, cov = eng.posterior_qbatch(c["xq"], q)
        d = eng.posterior_qbatch_grad(c["xq"], q, gm, gc)
        for lo, hi in ((0, 50), (1, 44), (6840, 6860), (163 * 42 - 1, 163 * 42 + 1), (b - 30, b)):
            sub = slice(lo * q, hi * q)
            smean, scov = eng.posterior_qbatch(c["xq"][sub], q)
            sd = eng.posterior_qbatch_grad(c["xq"][sub], q, gm[lo:hi], gc[lo:hi])
            assert np.array_equal(smean, mean[lo:hi]) and np.array_equal(scov, cov[lo:hi]), (lo, hi)
            assert np.array_equal(sd, d[sub]), (lo, hi)
        # device-resident inputs and outputs take the same path
        xd = torch.from_numpy(c["xq"][:300]).cuda()
        dmean, dcov = (torch.empty(s, dtype=torch.float64, device="cuda") for s in ((100, q), (100, q, q)))
        eng.posterior_qbatch(xd, q, out_mean=dmean, out_cov=dcov)
        dd = eng.posterior_qbatch_grad(xd, q, torch.from_numpy(gm[:100]).cuda(), torch.from_numpy(gc[:100]).cuda(),
                                       out=torch.empty(300, 32, dtype=torch.float64, device="cuda"))
        assert np.array_equal(dmean.cpu().numpy(), mean[:100]) and np.array_equal(dcov.cpu().numpy(), cov[:100])
        assert np.array_equal(dd.cpu().numpy(), d[:300])
    finally:
        eng.close()


def test_gradient_matches_central_differences():
    p = make_problem(200, 3, 2, dz=2, n_combo=3, n_noise=2, n_mean=2, seed=21)
    h = make_hyper(p, seed=11, noise=1e-2)
    q, b = 4, 3
    c = make_candidates(p, b * q, seed=22)
    gm, gc = _upstream(b, q, seed=23)
    eng = _engine(p)
    try:
        eng.factorize(h)
        d = eng.posterior_qbatch_grad(c["xq"], q, gm, gc, **_kw(c, True))

        def f(x):
            mean, cov = eng.posterior_qbatch(x, q, **_kw(c, True))
            return float((gm * mean).sum() + (gc * cov).sum())

        eps = 1e-5
        fd = np.zeros_like(d)
        for i in range(b * q):
            for k in range(p["dq"]):
                xp, xm = c["xq"].copy(), c["xq"].copy()
                xp[i, k] += eps
                xm[i, k] -= eps
                fd[i, k] = (f(xp) - f(xm)) / (2 * eps)
        only_mean = eng.posterior_qbatch_grad(c["xq"], q, gm, None, **_kw(c, True))
        only_cov = eng.posterior_qbatch_grad(c["xq"], q, None, gc, **_kw(c, True))
        assert np.count_nonzero(eng.posterior_qbatch_grad(c["xq"], q, None, None, **_kw(c, True))) == 0
    finally:
        eng.close()
    print("d_xq vs central differences: %.2e" % float(np.max(np.abs(d - fd))))
    np.testing.assert_allclose(d, fd, rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(only_mean + only_cov, d, rtol=1e-12, atol=1e-13)


def test_argument_checks():
    p = make_problem(100, 2, 0, seed=24)
    eng = _engine(p)
    try:
        eng.factorize(make_hyper(p, seed=1))
        x = make_candidates(p, 129 * 2, seed=25)["xq"]
        with pytest.raises(ValueError, match="GPP_MAX_QBATCH"):
            eng.posterior_qbatch(x, 129)
        with pytest.raises(ValueError, match="GPP_MAX_QBATCH"):
            eng.posterior_qbatch_grad(x, 129, None, np.zeros((2, 129, 129)))
        mean, cov = eng.posterior_qbatch(x[:0], 4)
        assert mean.shape == (0, 4) and cov.shape == (0, 4, 4)
    finally:
        eng.close()


def test_qei_lbfgsb_through_the_model():
    """Monte-Carlo qEI of b = 4 starts of q = 3 points, written in torch on GPR.posterior([b, q, d]) with fixed base
    samples, maximised by L-BFGS-B with the engine's gradient."""
    from scipy.optimize import minimize
    from gpplus_b200.models import GP_Plus
    rng = np.random.default_rng(26)
    X = rng.uniform(-2, 2, (80, 3))
    y = np.sin(X[:, 0]) + 0.5 * np.cos(1.5 * X[:, 1]) + 0.2 * X[:, 2] + 0.02 * rng.standard_normal(80)
    m = GP_Plus(torch.tensor(X), torch.tensor(y), dtype=torch.float64, quant_correlation_class="Matern52Kernel")
    with torch.no_grad():
        m.covar_module.raw_outputscale.fill_(0.5)
    b, q, S = 4, 3, 256
    E = torch.randn(S, b, q, generator=torch.Generator().manual_seed(3), dtype=torch.float64)
    best = float(np.quantile((y - float(m.y_min)) / float(m.y_std), 0.75))  # in the scaled units of posterior

    def qei(x):  # per-start values [b]
        post = m.posterior(x, observation_noise=False)
        f = post.rsample(torch.Size([S]), base_samples=E)
        return (f - best).clamp_min(0).max(-1).values.mean(0)

    def neg(flat):
        x = torch.tensor(flat.reshape(b, q, 3), requires_grad=True)
        v = qei(x).sum()
        g, = torch.autograd.grad(v, x)
        return -float(v.detach()), -g.numpy().reshape(-1)

    x0 = rng.uniform(-2, 2, (b, q, 3))
    val, grad = neg(x0.reshape(-1))
    eps = 1e-6
    for k in range(0, b * q * 3, 5):
        xp, xm = x0.reshape(-1).copy(), x0.reshape(-1).copy()
        xp[k] += eps
        xm[k] -= eps
        fd = (neg(xp)[0] - neg(xm)[0]) / (2 * eps)
        assert abs(fd - grad[k]) <= 1e-5 * max(1.0, abs(grad[k])), (k, fd, grad[k])
    res = minimize(neg, x0.reshape(-1), jac=True, method="L-BFGS-B", bounds=[(-2, 2)] * (b * q * 3),
                   options={"maxiter": 30})
    with torch.no_grad():
        before = qei(torch.tensor(x0))
        after = qei(torch.tensor(res.x.reshape(b, q, 3)))
    print("qEI before", before.numpy(), "after", after.numpy())
    assert bool((after > before).all()), (before, after)
    m.release_engine()
