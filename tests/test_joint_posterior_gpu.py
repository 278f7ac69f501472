"""gpp_predict_joint / gpp_sample_posterior on the B200: the joint predictive covariance against the dense CPU oracle
(tests/joint_posterior_reference.py), its agreement with gpp_predict, chunk stitching, the factor behind the draws,
the untouched handle state, and GP_Plus.predict_joint / sample_posterior end to end."""
import numpy as np
import pytest
import torch

from problems import engine_kwargs, make_candidates, make_hyper, make_problem

pytestmark = pytest.mark.gpu

# |Sigma_engine - Sigma_ref| per entry, relative to sigma_f^2; the bound leaves room for the INT8-sliced factor of K_y,
# which feeds U.  Worst case observed on one B200 (1000 W power limit): 2.3e-12 with the INT8-sliced factor at
# N = 3200, at most 1.7e-14 on every DMMA case, 1.8e-15 at model level.
COV_TOL = 1e-9


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


def _check(p, h, c, include_noise=False, fp64=None):
    from joint_posterior_reference import predict_joint as reference_predict_joint
    eng = _engine(p, fp64)
    try:
        eng.factorize(h)
        kw = _kw(c, include_noise)
        mu, cov = eng.predict_joint(c["xq"], **kw)
        mu0, var0 = eng.predict(c["xq"], min_var=1e-10, **kw)
        again = eng.predict_joint(c["xq"], **kw)
    finally:
        eng.close()
    sf2 = h["sigma_f2"]
    assert cov.shape == (c["m"], c["m"]) and np.all(np.isfinite(cov))
    assert np.array_equal(mu, mu0), "mean is not bitwise gpp_predict's"
    assert np.array_equal(cov, cov.T), "covariance is not exactly symmetric"
    assert np.array_equal(mu, again[0]) and np.array_equal(cov, again[1]), "repeated calls differ"
    free = var0 > 1e-10
    assert np.max(np.abs(np.diag(cov) - var0)[free], initial=0.0) <= 1e-12 * sf2
    rmu, rcov = reference_predict_joint(p, h, c, include_noise)
    err = float(np.max(np.abs(cov - rcov))) / sf2
    print("cov err %.2e (sigma_f^2 units)" % err)
    assert err <= COV_TOL, err
    assert np.max(np.abs(mu - rmu)) <= 1e-8
    return mu, cov


@pytest.mark.parametrize("kernel", [0, 1, 2])
@pytest.mark.parametrize("n", [1, 127, 129, 300])
def test_covariance_matches_oracle(kernel, n):
    p = make_problem(n, 4, kernel, seed=n + kernel)
    _check(p, make_hyper(p, seed=3), make_candidates(p, 129, seed=5))


@pytest.mark.parametrize("m", [1, 127, 128, 129, 300])
def test_candidate_counts(m):
    p = make_problem(300, 4, 0, seed=21)
    _check(p, make_hyper(p, seed=4), make_candidates(p, m, seed=m))


@pytest.mark.parametrize("n_pass", [1, 3])
def test_latent_map_and_ensemble(n_pass):
    p = make_problem(260, 3, 2, dz=2, n_combo=6, n_pass=n_pass, seed=11)
    _check(p, make_hyper(p, seed=4), make_candidates(p, 200, seed=6))


@pytest.mark.parametrize("include_noise", [False, True])
def test_noise_groups_and_means_with_zero_mean_group(include_noise):
    p = make_problem(300, 5, 0, dz=2, n_combo=4, n_noise=3, n_mean=3, zero_mean_group=True, seed=12)
    c = make_candidates(p, 257, seed=7)
    assert c["mean_idx"].min() == -1
    _check(p, make_hyper(p, seed=5, noise=1e-2), c, include_noise=include_noise)


@pytest.mark.parametrize("dq", [0, 32])
def test_input_widths(dq):
    if dq == 0:
        p = make_problem(200, 0, 0, dz=2, n_combo=5, seed=14)
        h = make_hyper(p, seed=7)
    else:
        p = make_problem(400, 32, 1, seed=13)
        h = make_hyper(p, seed=6, w_scale=0.02)
    _check(p, h, make_candidates(p, 150, seed=8))


@pytest.mark.parametrize("fp64", ["dmma", "int8"])
def test_int8_sliced_factor(fp64):
    from gpplus_b200 import _engine as E
    p = make_problem(3200, 4, 2, seed=15)
    _check(p, make_hyper(p, seed=8, noise=1e-3), make_candidates(p, 300, seed=10),
           fp64=E.FP64_DMMA if fp64 == "dmma" else E.FP64_INT8)


def test_chunks_stitch_bitwise_and_the_cap():
    """N = 9000: the K* chunk holds 14 720 candidates, so m = 16 384 crosses a chunk boundary.  Blocks of the joint
    covariance equal the joint covariance of the sub-batch alone, bitwise."""
    from gpplus_b200 import _engine as E
    p = make_problem(9000, 4, 0, seed=31)
    h = make_hyper(p, seed=12, noise=1e-2)
    c = make_candidates(p, E.MAX_JOINT, seed=13)
    eng = _engine(p)
    try:
        eng.factorize(h)
        mu, cov = eng.predict_joint(c["xq"])
        mu0, _ = eng.predict(c["xq"])
        assert np.array_equal(mu, mu0)
        for lo, hi in ((0, 300), (14592, 15000), (14080, 14848), (16384 - 640, 16384)):
            smu, scov = eng.predict_joint(c["xq"][lo:hi])
            assert np.array_equal(smu, mu[lo:hi])
            assert np.array_equal(scov, cov[lo:hi, lo:hi]), (lo, hi)
        del cov
        with pytest.raises(ValueError, match="GPP_MAX_JOINT"):
            eng.predict_joint(make_candidates(p, E.MAX_JOINT + 1, seed=14)["xq"])
        with pytest.raises(ValueError, match="GPP_MAX_JOINT"):
            eng.sample_posterior(c["xq"][:1].repeat(E.MAX_JOINT + 1, 0), np.zeros((1, E.MAX_JOINT + 1)))
    finally:
        eng.close()


@pytest.mark.parametrize("fp64", ["dmma", "int8"])
def test_identity_base_samples_recover_the_factor(fp64):
    from gpplus_b200 import _engine as E
    p = make_problem(3200 if fp64 == "int8" else 300, 4, 1, seed=17)
    h = make_hyper(p, seed=9, noise=1e-3)
    c = make_candidates(p, 300, seed=18)
    eng = _engine(p, E.FP64_DMMA if fp64 == "dmma" else E.FP64_INT8)
    try:
        eng.factorize(h)
        mu, cov = eng.predict_joint(c["xq"])
        draws, jit = eng.sample_posterior(c["xq"], np.eye(c["m"]))
    finally:
        eng.close()
    L = (draws - mu[None, :]).T  # draws[s, i] = mu_i + L[i, s]
    assert np.count_nonzero(np.triu(L, 1)) == 0
    assert np.all(np.diag(L) > 0)
    err = float(np.max(np.abs(L @ L.T - (cov + jit * np.eye(c["m"]))))) / h["sigma_f2"]
    print("jitter %g, |L L^T - (cov + jitter I)| %.2e sigma_f^2" % (jit, err))
    assert err <= 1e-12


@pytest.mark.parametrize("sizes", [(500, 300), (640, 500), (1100, 1000, 129)])
def test_repeated_sampling_with_fewer_candidates(sizes):
    """One handle, several gpp_sample_posterior calls with decreasing m: every call equals the same call on a fresh
    handle bitwise (the buffers of an earlier, larger call are read at another leading dimension)."""
    p = make_problem(400, 4, 2, seed=32)
    h = make_hyper(p, seed=15, noise=1e-3)
    c = make_candidates(p, max(sizes), seed=33)
    eng = _engine(p)
    try:
        eng.factorize(h)
        out = []
        for m in sizes:
            mu, cov = eng.predict_joint(c["xq"][:m])
            out.append((mu, cov) + eng.sample_posterior(c["xq"][:m], np.eye(m)))
    finally:
        eng.close()
    for m, (mu, cov, draws, jit) in zip(sizes, out):
        fresh = _engine(p)
        try:
            fresh.factorize(h)
            ref, rjit = fresh.sample_posterior(c["xq"][:m], np.eye(m))
        finally:
            fresh.close()
        assert jit == rjit and np.array_equal(draws, ref), m
        L = (draws - mu[None, :]).T
        err = float(np.max(np.abs(L @ L.T - (cov + jit * np.eye(m))))) / h["sigma_f2"]
        assert err <= 1e-12, (m, err)


def test_draws_have_the_posterior_covariance():
    p = make_problem(400, 3, 0, seed=19)
    h = make_hyper(p, seed=10, noise=1e-2, w_scale=1.0)
    c = make_candidates(p, 50, seed=20)
    S = 20000
    E_ = np.random.default_rng(21).standard_normal((S, c["m"]))
    eng = _engine(p)
    try:
        eng.factorize(h)
        mu, cov = eng.predict_joint(c["xq"])
        draws, jit = eng.sample_posterior(c["xq"], E_)
        again, _ = eng.sample_posterior(c["xq"], E_)
    finally:
        eng.close()
    assert jit == 0.0 and np.array_equal(draws, again)
    D = draws - mu[None, :]
    C = D.T @ D / S
    d = np.diag(cov)
    bound = 5.0 * np.sqrt((cov ** 2 + np.outer(d, d)) / S)
    assert np.all(np.abs(C - cov) <= bound), float(np.max(np.abs(C - cov) / bound))


def test_duplicate_candidates_take_the_oracle_jitter():
    """Two candidates on the same point make the joint covariance singular: the ladder reports the jitter that
    psd_safe_cholesky reports for the same matrix, and the two draws differ by O(sqrt(jitter))."""
    from joint_posterior_reference import joint_factor
    p = make_problem(300, 3, 0, seed=22)
    h = make_hyper(p, seed=11, noise=1e-3)
    c = make_candidates(p, 40, seed=23)
    c["xq"][1] = c["xq"][0]
    eng = _engine(p)
    try:
        eng.factorize(h)
        mu, cov = eng.predict_joint(c["xq"])
        draws, jit = eng.sample_posterior(c["xq"], np.random.default_rng(24).standard_normal((64, c["m"])))
    finally:
        eng.close()
    _, jit_ref = joint_factor(cov)
    print("engine jitter %g, psd_safe_cholesky on the same matrix %g" % (jit, jit_ref))
    assert jit == jit_ref
    gap = float(np.max(np.abs(draws[:, 0] - draws[:, 1])))
    assert gap <= 20.0 * np.sqrt(max(jit, 1e-16)), gap


def test_handle_state_is_untouched():
    from gpplus_b200 import _engine as E
    p = make_problem(500, 4, 2, dz=2, n_combo=3, n_noise=2, n_mean=2, seed=25)
    h = make_hyper(p, seed=13, noise=1e-2)
    c = make_candidates(p, 200, seed=26)
    eng = _engine(p)
    try:
        with pytest.raises(ValueError, match="gpp_factorize"):
            eng.predict_joint(c["xq"], **_kw(c, False))
        with pytest.raises(ValueError, match="gpp_factorize"):
            eng.sample_posterior(c["xq"], np.zeros((2, c["m"])), **_kw(c, False))
        eng.mll_grad(h, want_grad=True)

        def state():
            return ([eng.fetch(k) for k in ("L", "Linv", "Kinv", "alpha")] + list(eng.predict(c["xq"], **_kw(c, True))),
                    eng.stats(), eng.timings())

        before = state()
        eng.predict_joint(c["xq"], **_kw(c, True))
        mid = state()
        eng.sample_posterior(c["xq"], np.ones((3, c["m"])), **_kw(c, True))
        after = state()
    finally:
        eng.close()
    for s in (mid, after):
        assert all(np.array_equal(a, b) for a, b in zip(before[0], s[0]))
        assert before[1] == s[1] and before[2] == s[2]


def test_prediction_launches_are_unchanged():
    """gpp_predict / gpp_predict_grad / gpp_acq_argmax issue the launches they issued before the joint entries were
    added: prep + n_pass covariance launches + K* L^-T + finish per chunk (+ V, gradient tiles and their finish)."""
    from gpplus_b200 import _engine as E
    p = make_problem(300, 4, 0, dz=2, n_combo=3, n_pass=2, seed=27)
    c = make_candidates(p, 500, seed=28)
    eng = _engine(p)
    try:
        eng.factorize(make_hyper(p, seed=14))
        counts = []
        for call in (lambda: eng.predict(c["xq"], level_idx=c["level_idx"]),
                     lambda: eng.predict_grad(c["xq"], level_idx=c["level_idx"]),
                     lambda: eng.acq_argmax(c["xq"], None, [1.0], [E.ACQ_EI], [0.5], level_idx=c["level_idx"])):
            k0 = E.launch_count()
            call()
            counts.append(E.launch_count() - k0)
        k0 = E.launch_count()
        eng.predict_joint(c["xq"], level_idx=c["level_idx"])
        joint = E.launch_count() - k0
    finally:
        eng.close()
    assert counts == [3 + 2, 6 + 2, 3 + 2], counts
    # J1: one prep + the predict chunk without its prep; J2: diagonal, n_pass covariance launches, SYRK; mirror
    assert joint == 1 + (2 + 2) + (1 + 2 + 1) + 1, joint


def test_model_level_against_dense_reference():
    import test_model_gpu as TM
    from gpplus_b200._dense import dense_model_covariance
    m, _, Xte, _ = TM._c2()
    Xq = Xte[:60].clone()
    mean, cov = m.predict_joint(Xq)
    m.eval()
    Xtr = m.train_inputs[0]
    n = Xtr.shape[0]
    with torch.no_grad():
        K = dense_model_covariance(m, torch.cat([Xtr, Xq], 0))
        noise = m.likelihood.noise.reshape(-1).double()
        Ky = K[:n, :n] + noise[0] * torch.eye(n, dtype=torch.float64)
        L = torch.linalg.cholesky(Ky)
        V = torch.linalg.solve_triangular(L, K[:n, n:], upper=False)
        ref = (K[n:, n:] - V.T @ V) * m.y_std.double() ** 2
        sf2 = float(m.covar_module.outputscale)
    err = float((cov - ref).abs().max()) / (sf2 * float(m.y_std) ** 2)
    print("model-level cov err %.2e" % err)
    assert err <= 1e-9
    mean0, std0 = m.predict(Xq, return_std=True, include_noise=False)
    assert torch.equal(mean, mean0)
    draws = m.sample_posterior(Xq, num_samples=20000, generator=torch.Generator().manual_seed(5))
    assert draws.shape == (20000, Xq.shape[0])
    sd = draws.std(0)
    # the standard deviation of a sample standard deviation is about sigma / sqrt(2 S)
    assert torch.all((sd - std0).abs() <= 5.0 * std0 / np.sqrt(2 * 20000) + 1e-12)
