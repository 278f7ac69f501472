"""gpp_gibbon_qbatch and gpp_max_value_quartiles on the B200: GIBBON values and input gradients against torch on the
engine's own latent t-batch posteriors and against the dense CPU reference (tests/gibbon_reference.py), bitwise
identities (repeated, values-only, sub-ranges across chunk boundaries, device-resident), the projected identity, the
per-t-batch jitter, the untouched handle, argument and status codes, the max-value quartiles against the torch
bisection, and multi-fidelity GIBBON end to end."""
import numpy as np
import pytest
import torch

from gibbon_reference import gibbon_block, gibbon_qbatch as reference_gibbon, max_value_quartiles, row_noise
from problems import engine_kwargs, make_candidates, make_hyper, make_problem
from qacq_reference import ladder_jitter

pytestmark = pytest.mark.gpu

VAL_TOL_ENGINE = 1e-9  # |v - v_torch| on the engine's own blocks, nats
VAL_TOL_DENSE = 1e-8   # |v - v_ref| against the dense CPU reference, nats
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


def _max_values(mean, k, maximize, seed=0):
    """k values around and above the largest sigma mu (scaled units)."""
    sgn = 1.0 if maximize else -1.0
    top = float(np.max(sgn * mean))
    return top + np.abs(np.random.default_rng(seed).standard_normal(k)) * 0.3 - 0.05


def _check(p, h, c, q, projected, k=10, fp64=None, maximize=True, dense=True):
    q_tot = 2 * q if projected else q
    b = c["m"] // q_tot
    kw = _kw(c)
    eng = _engine(p, fp64)
    try:
        eng.factorize(h)
        mu0, var0 = eng.predict(c["xq"], min_var=-np.inf, **kw)
        alpha0, stats0 = eng.fetch("alpha"), eng.stats()
        mean, cov = eng.posterior_qbatch(c["xq"], q_tot, include_noise=False, **kw)
        mv = _max_values(mean, k, maximize, seed=q_tot)
        v, d, jit = eng.gibbon_qbatch(c["xq"], q, mv, projected=projected, maximize=maximize, **kw)
        v1, d1, jit1 = eng.gibbon_qbatch(c["xq"], q, mv, projected=projected, maximize=maximize, **kw)
        v0, none, jit0 = eng.gibbon_qbatch(c["xq"], q, mv, projected=projected, maximize=maximize, want_grad=False,
                                           **kw)
        noise = row_noise(h, c, q_tot, q)
        vt, gm, gc, _ = gibbon_block(mean, cov, noise, q, projected, mv, maximize, jit)
        d_eng = eng.posterior_qbatch_grad(c["xq"], q_tot, gm, gc, include_noise=False, **kw)
        mu1, var1 = eng.predict(c["xq"], min_var=-np.inf, **kw)
        assert np.array_equal(eng.fetch("alpha"), alpha0) and np.array_equal(mu1, mu0) and np.array_equal(var1, var0)
        assert eng.stats() == stats0
    finally:
        eng.close()
    assert v.shape == (b,) and d.shape == (b * q_tot, p["dq"]) and jit.shape == (b,) and none is None
    assert np.all(np.isfinite(v)) and np.all(np.isfinite(d))
    assert np.array_equal(v, v1) and np.array_equal(d, d1) and np.array_equal(jit, jit1), "repeated calls differ"
    assert np.array_equal(v0, v) and np.array_equal(jit0, jit), "values-only differs from the gradient call"
    V = cov[:, :q, :q] + np.stack([np.diag(n) for n in noise])
    np.testing.assert_array_equal(jit, ladder_jitter(torch.from_numpy(V)).numpy())
    verr = float(np.max(np.abs(v - vt)))
    scale = max(1.0, float(np.max(np.abs(d_eng), initial=0.0)))
    derr = float(np.max(np.abs(d - d_eng), initial=0.0)) / scale
    print("q=%d projected=%d K=%d b=%d jitter %.0e: engine blocks value %.2e d_xq %.2e"
          % (q, projected, k, b, float(jit.max()), verr, derr))
    assert verr <= VAL_TOL_ENGINE, verr
    assert derr <= GRAD_TOL, derr
    if dense:
        rv, rd, _ = reference_gibbon(p, h, c, q, projected, mv, maximize, jit)
        rverr = float(np.max(np.abs(v - rv)))
        rderr = float(np.max(np.abs(d - rd), initial=0.0)) / max(1.0, float(np.max(np.abs(rd), initial=0.0)))
        print("   dense reference: value %.2e d_xq %.2e" % (rverr, rderr))
        assert rverr <= VAL_TOL_DENSE, rverr
        assert rderr <= GRAD_TOL, rderr
    return v, d, jit


@pytest.mark.parametrize("kernel", [0, 1, 2])
@pytest.mark.parametrize("q,projected", [(1, 0), (1, 1), (4, 0), (4, 1), (16, 0), (16, 1), (64, 0), (64, 1)])
@pytest.mark.parametrize("k", [1, 10, 1000])
def test_kernels_batch_shapes_and_samples(kernel, q, projected, k):
    p = make_problem(300, 4, kernel, seed=kernel + 1)
    q_tot = 2 * q if projected else q
    b = max(2, 256 // q_tot)
    _check(p, make_hyper(p, seed=3, noise=1e-2), make_candidates(p, b * q_tot, seed=q_tot), q, bool(projected), k,
           maximize=(kernel + k) % 2 == 0, dense=q_tot <= 32)


@pytest.mark.parametrize("maximize", [True, False])
@pytest.mark.parametrize("projected", [False, True])
def test_mixed_variables_noise_groups_means_and_latent_source(maximize, projected):
    """The source is a latent categorical (level_idx) with its own noise group and mean; the target rows carry the
    target source's level, noise group and mean."""
    p = make_problem(300, 3, 1, dz=2, n_combo=4, n_noise=3, n_mean=3, zero_mean_group=True, seed=12)
    h = make_hyper(p, seed=5, noise=1e-2)
    q, b = 3, 30
    c = make_candidates(p, b * (2 * q if projected else q), seed=7)
    if projected:
        for key in ("level_idx", "noise_idx", "mean_idx"):
            a = c[key].reshape(b, 2 * q)
            a[:, q:] = 0
            c[key] = np.ascontiguousarray(a.reshape(-1))
        xq = c["xq"].reshape(b, 2 * q, -1)
        xq[:, q:] = xq[:, :q]
        c["xq"] = np.ascontiguousarray(xq.reshape(b * 2 * q, -1))
    _check(p, h, c, q, projected, 10, maximize=maximize)


@pytest.mark.parametrize("fp64", ["dmma", "int8"])
def test_int8_sliced_factor(fp64):
    from gpplus_b200 import _engine as E
    p = make_problem(3200, 4, 2, seed=15)
    _check(p, make_hyper(p, seed=8, noise=1e-2), make_candidates(p, 40 * 8, seed=10), 4, True, 10,
           fp64=E.FP64_DMMA if fp64 == "dmma" else E.FP64_INT8)


def test_other_batches_and_chunk_split_do_not_matter():
    """N = 3200, dq = 32, q_tot = 2: chunks of 163 tiles of 64 t-batches, so the call takes three chunks.  Any run of
    t-batches called alone gives bitwise the full call's values, jitters and gradients, and so do device-resident
    inputs and outputs."""
    p = make_problem(3200, 32, 2, n_noise=2, n_mean=2, seed=18)
    h = make_hyper(p, seed=10, noise=1e-3, w_scale=0.02)
    q, b = 1, 163 * 64 * 2 + 17
    c = make_candidates(p, b * 2, seed=19)
    kw = _kw(c)
    mv = np.array([1.1, 1.3, 0.9])
    eng = _engine(p)
    try:
        eng.factorize(h)
        v, d, jit = eng.gibbon_qbatch(c["xq"], q, mv, projected=True, **kw)
        for lo, hi in ((0, 50), (1, 44), (10400, 10450), (163 * 64 - 1, 163 * 64 + 1), (b - 30, b)):
            sub = slice(lo * 2, hi * 2)
            sub_kw = {k: None if a is None else a[sub] for k, a in kw.items()}
            sv, sd, sj = eng.gibbon_qbatch(c["xq"][sub], q, mv, projected=True, **sub_kw)
            assert np.array_equal(sv, v[lo:hi]) and np.array_equal(sj, jit[lo:hi]), (lo, hi)
            assert np.array_equal(sd, d[sub]), (lo, hi)
        dev = {k: None if a is None else torch.from_numpy(a[:200]).cuda() for k, a in kw.items()}
        xd = torch.from_numpy(c["xq"][:200]).cuda()
        vd = torch.empty(100, dtype=torch.float64, device="cuda")
        dd = torch.empty(200, 32, dtype=torch.float64, device="cuda")
        eng.gibbon_qbatch(xd, q, torch.from_numpy(mv).cuda(), projected=True, out_values=vd, out_d_xq=dd, **dev)
        assert np.array_equal(vd.cpu().numpy(), v[:100]) and np.array_equal(dd.cpu().numpy(), d[:200])
    finally:
        eng.close()


def test_projected_identity():
    """Target rows equal to the actual rows (same inputs, levels and means) give the unprojected values and, folded,
    the unprojected gradients."""
    p = make_problem(300, 3, 2, n_noise=2, n_mean=2, seed=40)
    q, b = 3, 20
    c = make_candidates(p, b * q, seed=41)
    kw = _kw(c)

    def doubled(a):
        a = a.reshape(b, q, -1)
        return np.ascontiguousarray(np.concatenate([a, a], 1).reshape(b * 2 * q, *a.shape[2:]).squeeze())

    c2 = {k: doubled(c[k]) if c.get(k) is not None else None for k in ("xq", "level_idx", "noise_idx", "mean_idx")}
    c2["xq"] = c2["xq"].reshape(b * 2 * q, -1)
    eng = _engine(p)
    try:
        eng.factorize(make_hyper(p, seed=14, noise=1e-2))
        for maximize in (True, False):
            mv = np.array([0.8, 1.2]) if maximize else np.array([0.1, -0.2])
            v0, d0, _ = eng.gibbon_qbatch(c["xq"], q, mv, maximize=maximize, **kw)
            v1, d1, _ = eng.gibbon_qbatch(c2["xq"], q, mv, projected=True, maximize=maximize, level_idx=c2["level_idx"],
                                          noise_idx=c2["noise_idx"], mean_idx=c2["mean_idx"])
            d1 = d1.reshape(b, 2 * q, -1)
            fold = (d1[:, :q] + d1[:, q:]).reshape(b * q, -1)
            verr = float(np.max(np.abs(v0 - v1)))
            derr = float(np.max(np.abs(d0 - fold))) / max(1.0, float(np.max(np.abs(d0))))
            print("projected identity: value %.2e d_xq %.2e" % (verr, derr))
            assert verr <= 1e-12 and derr <= 1e-12
    finally:
        eng.close()


def test_gradient_matches_central_differences():
    p = make_problem(200, 3, 2, dz=2, n_combo=3, n_noise=2, n_mean=2, seed=21)
    h = make_hyper(p, seed=11, noise=1e-2)
    q, b = 2, 3
    c = make_candidates(p, b * 2 * q, seed=22)
    kw = _kw(c)
    mv = np.array([1.0, 1.2, 1.5])
    eng = _engine(p)
    try:
        eng.factorize(h)
        _, d, _ = eng.gibbon_qbatch(c["xq"], q, mv, projected=True, **kw)

        def f(x):
            return float(eng.gibbon_qbatch(x, q, mv, projected=True, want_grad=False, **kw)[0].sum())

        eps = 1e-6
        fd = np.zeros_like(d)
        for i in range(b * 2 * q):
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
    """t-batch 1 repeats one point far from every training point in a noise group without noise: V is exactly the
    all-ones matrix and the ladder gives 1e-8; the other t-batches take none."""
    p = make_problem(200, 3, 0, n_noise=2, seed=32)
    p["noise_idx"] = np.zeros(200, dtype=np.int32)
    q, b = 6, 4
    c = make_candidates(p, b * q, seed=33)
    c["noise_idx"] = np.zeros(b * q, dtype=np.int32)
    c["xq"][q:2 * q] = 1e3
    c["noise_idx"][q:2 * q] = 1
    h = make_hyper(p, seed=13, noise=1e-4)
    h["sigma_f2"] = 1.0
    h["noise"] = np.array([1e-4, 0.0])
    mv = np.array([1.0, 1.3])
    eng = _engine(p)
    try:
        eng.factorize(h)
        mean, cov = eng.posterior_qbatch(c["xq"], q, **_kw(c))
        v, d, jit = eng.gibbon_qbatch(c["xq"], q, mv, **_kw(c))
    finally:
        eng.close()
    assert np.array_equal(cov[1], np.ones((q, q)))
    noise = row_noise(h, c, q, q)
    V = cov + np.stack([np.diag(n) for n in noise])
    assert np.array_equal(jit, ladder_jitter(torch.from_numpy(V)).numpy()) and np.array_equal(jit, [0, 1e-8, 0, 0])
    vt, _, _, _ = gibbon_block(mean, cov, noise, q, False, mv, True, jit)
    tol = [VAL_TOL_ENGINE, 1e-6, VAL_TOL_ENGINE, VAL_TOL_ENGINE]  # pivots of 1e-8 carry eps / 1e-8 rounding
    print("jitter", jit, "value vs torch", np.abs(v - vt))
    assert np.all(np.abs(v - vt) <= tol) and np.all(np.isfinite(d))


def test_argument_and_status_codes():
    from gpplus_b200 import _engine as E
    p = make_problem(100, 2, 0, seed=24)
    x4, mv4, q3, v4 = np.zeros((4, 2)), np.array([1.0]), np.empty(3), np.empty(4)
    lib = E.load_library()
    # a null handle, and a handle whose factor is not formed yet
    assert lib.gpp_gibbon_qbatch(None, 4, 1, 0, E._ptr(x4), None, None, None, 1, 1, E._ptr(mv4), E._ptr(v4), None,
                                 None) == E.GPP_ERR_ARG
    assert lib.gpp_max_value_quartiles(None, 4, E._ptr(x4), None, None, 1, E._ptr(q3)) == E.GPP_ERR_ARG
    eng = _engine(p)
    try:
        rc = lib.gpp_gibbon_qbatch(eng._h, 4, 1, 0, E._ptr(x4), None, None, None, 1, 1, E._ptr(mv4), E._ptr(v4), None,
                                   None)
        assert rc == E.GPP_ERR_ARG and b"gpp_factorize" in lib.gpp_last_error()
        rc = lib.gpp_max_value_quartiles(eng._h, 4, E._ptr(x4), None, None, 1, E._ptr(q3))
        assert rc == E.GPP_ERR_ARG and b"gpp_factorize" in lib.gpp_last_error()
    finally:
        eng.close()
    # dq > GPP_MAX_DQ: no handle of that width can be created, so neither entry can be reached with one
    with pytest.raises((ValueError, E.EngineError)):
        E.Engine(**engine_kwargs(make_problem(40, 33, 0, seed=3)))
    eng = _engine(p)
    try:
        eng.factorize(make_hyper(p, seed=1))
        x = np.ascontiguousarray(make_candidates(p, 129 * 2, seed=25)["xq"])
        mv = np.array([1.0, 1.2])
        vals = np.empty(2)
        lib, h = eng._lib, eng._h
        for b, q, pr, k, m_, out, match in ((2, 0, 0, 2, mv, vals, b"q must"), (2, 4, 2, 2, mv, vals, b"projected"),
                                            (2, 65, 1, 2, mv, vals, b"GPP_MAX_QBATCH"),
                                            (2, 129, 0, 2, mv, vals, b"GPP_MAX_QBATCH"),
                                            (-1, 4, 0, 2, mv, vals, b"b must"), (2, 4, 0, 0, mv, vals, b"n_max_values"),
                                            (2, 4, 0, 65537, mv, vals, b"n_max_values"),
                                            (2, 4, 0, 2, None, vals, b"missing"), (2, 4, 0, 2, mv, None, b"missing")):
            rc = lib.gpp_gibbon_qbatch(h, b, q, pr, E._ptr(x), None, None, None, 1, k, E._ptr(m_), E._ptr(out), None,
                                       None)
            assert rc == E.GPP_ERR_ARG and match in lib.gpp_last_error(), (b, q, pr, k)
        q3 = np.empty(3)
        for m_, out, match in ((0, q3, b"m must"), (4, None, b"missing")):
            rc = lib.gpp_max_value_quartiles(h, m_, E._ptr(x), None, None, 1, E._ptr(out))
            assert rc == E.GPP_ERR_ARG and match in lib.gpp_last_error()
        v, d, jit = eng.gibbon_qbatch(x[:0], 4, mv)
        assert v.shape == (0,) and jit.shape == (0,)
        xn = x[:16].copy()
        xn[9, 1] = np.nan
        with pytest.raises(Exception, match="NaN"):
            eng.gibbon_qbatch(xn, 4, mv)
        with pytest.raises(Exception, match="NaN"):
            eng.max_value_quartiles(xn)
    finally:
        eng.close()
    # two identical points far from the training set in a noise group of -1e-5: V = ones - 1e-5 I fails every rung
    p = make_problem(100, 2, 0, n_noise=2, seed=26)
    p["noise_idx"] = np.zeros(100, dtype=np.int32)
    h = make_hyper(p, seed=2)
    h["sigma_f2"] = 1.0
    h["noise"] = np.array([1e-3, -1e-5])
    c = make_candidates(p, 2 * 2, seed=27)
    c["xq"][:2] = 1e3
    c["noise_idx"] = np.array([1, 1, 0, 0], dtype=np.int32)
    eng = _engine(p)
    try:
        eng.factorize(h)
        with pytest.raises(Exception, match="not positive definite"):
            eng.gibbon_qbatch(c["xq"], 2, np.array([1.0]), noise_idx=c["noise_idx"])
    finally:
        eng.close()


@pytest.mark.parametrize("m", [1, 100_000, 2_000_000])
def test_max_value_quartiles_against_torch(m):
    """At m = 2e6 the candidates lie far from the data in one mean group, so every marginal is close to the prior's:
    the sum of 2e6 terms log Phi(5) is below log 3/4 and the bracket has to widen."""
    p = make_problem(300, 3, 2, n_mean=2, seed=60)
    c = make_candidates(p, m, seed=61)
    widen = m == 2_000_000
    if widen:
        c["xq"] = 50.0 + 0.01 * c["xq"]
        c["mean_idx"] = np.zeros(m, dtype=np.int32)
    eng = _engine(p)
    try:
        eng.factorize(make_hyper(p, seed=15, noise=1e-2))
        for maximize in (True, False):
            mean, var = eng.predict(c["xq"], mean_idx=c["mean_idx"], min_var=1e-8)
            qs = eng.max_value_quartiles(c["xq"], mean_idx=c["mean_idx"], maximize=maximize)
            qs2 = eng.max_value_quartiles(c["xq"], mean_idx=c["mean_idx"], maximize=maximize)
            out = torch.empty(3, dtype=torch.float64, device="cuda")
            eng.max_value_quartiles(torch.from_numpy(c["xq"]).cuda(), mean_idx=torch.from_numpy(c["mean_idx"]).cuda(),
                                    maximize=maximize, out=out)
            want, lo, hi = max_value_quartiles(mean, var, maximize)
            sgn, sd = (1.0 if maximize else -1.0), float(np.sqrt(var).max())
            first = float(np.max(sgn * mean)) - float(np.min(sgn * mean)) + 10.0 * sd
            assert (hi - lo > 1.5 * first) == widen
            err = float(np.max(np.abs(qs - want))) / (hi - lo)
            print("m=%d maximize=%d: quartiles %s, torch %s, |diff| / (hi - lo) %.2e, hi - lo %.3g"
                  % (m, maximize, qs, want, err, hi - lo))
            assert err <= 1e-9
            assert np.array_equal(qs, qs2) and np.array_equal(out.cpu().numpy(), qs)
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
    return GP_Plus(torch.tensor(X), torch.tensor(y), qual_dict={2: 2}, multiple_noise=True, dtype=torch.float64)


def test_multi_fidelity_gibbon_end_to_end():
    from gpplus_b200.bayesian_optimizations import optimize_gibbon
    m = _mf_model()
    bounds = np.array([[-2.0, -2.0], [2.0, 2.0]])
    target, cost = 0, {0: 10.0, 1: 1.0}
    cand = torch.zeros(4096, 3, dtype=torch.float64)
    cand[:, :2] = -2.0 + 4.0 * torch.quasirandom.SobolEngine(2, scramble=True, seed=1).draw(4096, dtype=torch.float64)
    with torch.no_grad():
        mu_max = float(m.predict(cand, return_std=False).max())
    for method in ("gumbel", "thompson"):
        mv = m.sample_max_values(cand, 16, method=method, seed=2)
        assert mv.shape == (16,) and bool(torch.isfinite(mv).all())
        assert torch.equal(mv, m.sample_max_values(cand, 16, method=method, seed=2))
        print("%s max values: median %.4f, largest mean %.4f" % (method, float(mv.median()), mu_max))
        assert float(mv.median()) > mu_max - 0.05
        tfc = {2: target}
        for args in (dict(sequential=True, sources=[0, 1], cost_by_source=cost), dict(sequential=False),
                     dict(sequential=True, cost_by_source=cost)):
            q = 2
            fixed = {} if "sources" in args else {2: 1}
            X, v = optimize_gibbon(m, bounds, q, mv, fixed_columns=fixed, target_fixed_columns=tfc, num_restarts=3,
                                   raw_samples=32, options={"maxiter": 20}, seed=4, **args)
            assert X.shape == (q, 3) and bool(torch.isfinite(X).all()) and bool((X[:, :2].abs() <= 2.0).all())
            if "sources" not in args:
                assert bool((X[:, 2] == 1).all())
            assert bool(torch.isin(X[:, 2], torch.tensor([0.0, 1.0])).all())
            with torch.no_grad():
                again = float(m.gibbon(X[None], mv, target_fixed_columns=tfc,
                                       cost_by_source=args.get("cost_by_source"))[0])
            print("%s %s: X %s value %.6g" % (method, args, X.tolist(), v))
            assert np.isfinite(v) and again == v
    m.release_engine()
