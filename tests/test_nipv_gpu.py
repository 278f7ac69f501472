"""gpp_ipv_points / gpp_nipv_qbatch on the B200: values and input gradients against the dense CPU reference
(tests/nipv_reference.py) across kernels, q, M, latent maps, noise groups, input widths and both FP64 arithmetics;
bitwise identities (repeated, values-only, sub-ranges across chunk boundaries, device-resident, untouched handle
state); stale integration sets; argument checks; central differences; and GPR.acquisition_qbatch(X, "qNIPV") /
optimize_acquisition_qbatch end to end."""
import numpy as np
import pytest
import torch

from nipv_reference import nipv_qbatch as reference_nipv, nipv_refit
from problems import engine_kwargs, make_candidates, make_hyper, make_problem

pytestmark = pytest.mark.gpu

VAL_TOL = 1e-8   # |v - v_ref|, scaled units
GRAD_TOL = 1e-7  # |d - d_ref| relative to the largest |d_ref|


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
    return dict(level_idx=c["level_idx"], noise_idx=c["noise_idx"])


def _check(p, h, c, ipv, q, fp64=None):
    b = c["m"] // q
    eng = _engine(p, fp64)
    try:
        eng.factorize(h)
        mu0, var0 = eng.predict(c["xq"], min_var=-np.inf, level_idx=c["level_idx"])
        alpha0, stats0, tm0 = eng.fetch("alpha"), eng.stats(), eng.timings()
        eng.ipv_points(ipv["xq"], level_idx=ipv["level_idx"])
        v, d, jit = eng.nipv_qbatch(c["xq"], q, **_kw(c))
        v1, d1, jit1 = eng.nipv_qbatch(c["xq"], q, **_kw(c))
        v0, none, jit0 = eng.nipv_qbatch(c["xq"], q, want_grad=False, **_kw(c))
        mu1, var1 = eng.predict(c["xq"], min_var=-np.inf, level_idx=c["level_idx"])
        assert np.array_equal(eng.fetch("alpha"), alpha0) and np.array_equal(mu1, mu0) and np.array_equal(var1, var0)
        assert eng.stats() == stats0 and eng.timings() == tm0
    finally:
        eng.close()
    assert v.shape == (b,) and d.shape == (b * q, p["dq"]) and jit.shape == (b,) and none is None
    assert np.all(np.isfinite(v)) and np.all(np.isfinite(d))
    assert np.array_equal(v, v1) and np.array_equal(d, d1) and np.array_equal(jit, jit1), "repeated calls differ"
    assert np.array_equal(v0, v) and np.array_equal(jit0, jit), "values-only differs from the gradient call"
    rv, rd, rj = reference_nipv(p, h, c, ipv, q, jitter=jit)
    verr = float(np.max(np.abs(v - rv)))
    derr = float(np.max(np.abs(d - rd), initial=0.0)) / max(1e-300, float(np.max(np.abs(rd), initial=1e-300)))
    print("q=%d M=%d b=%d jitter %.0e: value %.2e d_xq %.2e (relative)" % (q, ipv["m"], b, float(jit.max()), verr,
                                                                         derr))
    assert verr <= VAL_TOL, verr
    assert derr <= GRAD_TOL, derr
    return v, d, jit


@pytest.mark.parametrize("kernel", [0, 1, 2])
@pytest.mark.parametrize("q", [1, 3, 8, 64, 128])
def test_kernels_and_batch_sizes(kernel, q):
    p = make_problem(300, 4, kernel, seed=kernel + 1)
    b = max(2, 192 // q)
    _check(p, make_hyper(p, seed=3, noise=1e-2), make_candidates(p, b * q, seed=q), make_candidates(p, 200, seed=50),
           q)


@pytest.mark.parametrize("M", [1, 1000])
def test_integration_sizes(M):
    p = make_problem(300, 3, 2, seed=40)
    _check(p, make_hyper(p, seed=4, noise=1e-2), make_candidates(p, 12 * 4, seed=41), make_candidates(p, M, seed=42),
           4)


@pytest.mark.parametrize("n_pass", [1, 3])
def test_latent_map_and_noise_groups(n_pass):
    p = make_problem(260, 3, 2, dz=2, n_combo=6, n_noise=3, n_pass=n_pass, seed=11)
    _check(p, make_hyper(p, seed=4, noise=1e-2), make_candidates(p, 20 * 5, seed=6), make_candidates(p, 150, seed=7),
           5)


@pytest.mark.parametrize("dq", [0, 32])
def test_input_widths(dq):
    if dq == 0:
        p = make_problem(200, 0, 0, dz=2, n_combo=5, seed=14)
        h = make_hyper(p, seed=7, noise=1e-2)
    else:
        p = make_problem(400, 32, 2, seed=13)
        h = make_hyper(p, seed=6, noise=1e-2, w_scale=0.02)
    _check(p, h, make_candidates(p, 16 * 6, seed=8), make_candidates(p, 130, seed=9), 6)


@pytest.mark.parametrize("fp64", ["dmma", "int8"])
def test_int8_sliced_factor(fp64):
    from gpplus_b200 import _engine as E
    p = make_problem(3200, 4, 2, seed=15)
    _check(p, make_hyper(p, seed=8, noise=1e-2), make_candidates(p, 10 * 8, seed=10), make_candidates(p, 200, seed=11),
           8, fp64=E.FP64_DMMA if fp64 == "dmma" else E.FP64_INT8)


def test_chunk_cap_split_other_batches_and_device_inputs():
    """M = 16384 caps a chunk at 2^27 / 16384 = 8192 rows, 1024 t-batches of q = 8: 2053 t-batches take three chunks.
    Any run of t-batches called alone gives bitwise the full call's values, jitters and gradients, and so do
    device-resident inputs and outputs; t-batches on both sides of a boundary match botorch's refit semantics."""
    p = make_problem(300, 4, 2, n_noise=2, seed=18)
    h = make_hyper(p, seed=10, noise=1e-2)
    q, b = 8, 1024 * 2 + 5
    c = make_candidates(p, b * q, seed=19)
    ipv = make_candidates(p, 16384, seed=20)
    eng = _engine(p)
    try:
        eng.factorize(h)
        eng.ipv_points(ipv["xq"])
        v, d, jit = eng.nipv_qbatch(c["xq"], q, **_kw(c))
        for lo, hi in ((0, 50), (1, 44), (1023, 1025), (1000, 1100), (b - 30, b)):
            sub = slice(lo * q, hi * q)
            sv, sd, sj = eng.nipv_qbatch(c["xq"][sub], q, noise_idx=c["noise_idx"][sub])
            assert np.array_equal(sv, v[lo:hi]) and np.array_equal(sj, jit[lo:hi]), (lo, hi)
            assert np.array_equal(sd, d[sub]), (lo, hi)
        xd = torch.from_numpy(c["xq"][:400]).cuda()
        nd = torch.from_numpy(c["noise_idx"][:400]).cuda()
        vd = torch.empty(50, dtype=torch.float64, device="cuda")
        dd = torch.empty(400, 4, dtype=torch.float64, device="cuda")
        eng.nipv_qbatch(xd, q, noise_idx=nd, out_values=vd, out_d_xq=dd)
        assert np.array_equal(vd.cpu().numpy(), v[:50]) and np.array_equal(dd.cpu().numpy(), d[:400])
    finally:
        eng.close()
    pick = [0, 1023, 1024, 2048, b - 1]
    rows = np.concatenate([np.arange(t * q, (t + 1) * q) for t in pick])
    sub = {"m": len(rows), "xq": c["xq"][rows], "level_idx": None, "noise_idx": c["noise_idx"][rows]}
    ref = nipv_refit(p, h, sub, ipv, q)
    print("chunk split: refit semantics %.2e" % float(np.max(np.abs(v[pick] - ref))))
    np.testing.assert_allclose(v[pick], ref, rtol=0, atol=VAL_TOL)


def test_stale_sets_are_refused_and_a_new_set_matches_a_fresh_engine():
    from gpplus_b200 import _engine as E
    p = make_problem(150, 3, 1, seed=60)
    h, h2 = make_hyper(p, seed=1, noise=1e-2), make_hyper(p, seed=2, noise=1e-2)
    c, ipv = make_candidates(p, 6 * 3, seed=61), make_candidates(p, 40, seed=62)
    eng = _engine(p)
    try:
        eng.factorize(h)
        with pytest.raises(ValueError, match="integration set"):
            eng.nipv_qbatch(c["xq"], 3)
        eng.ipv_points(ipv["xq"])
        eng.nipv_qbatch(c["xq"], 3)
        eng.factorize(h2)
        with pytest.raises(ValueError, match="integration set"):
            eng.nipv_qbatch(c["xq"], 3)
        eng.mll_grad(h, want_grad=False)
        with pytest.raises(ValueError, match="integration set"):
            eng.nipv_qbatch(c["xq"], 3)
        eng.factorize(h2)
        eng.ipv_points(ipv["xq"])
        v, d, jit = eng.nipv_qbatch(c["xq"], 3)
    finally:
        eng.close()
    fresh = _engine(p)
    try:
        fresh.factorize(h2)
        fresh.ipv_points(ipv["xq"])
        fv, fd, fj = fresh.nipv_qbatch(c["xq"], 3)
    finally:
        fresh.close()
    assert np.array_equal(v, fv) and np.array_equal(d, fd) and np.array_equal(jit, fj)
    # a handle parked in the pool and handed back to the next engine of the same shape holds no set
    parked = _engine(p)
    parked.factorize(h)
    parked.close()
    again = _engine(p)
    try:
        again.factorize(h)
        with pytest.raises(ValueError, match="integration set"):
            again.nipv_qbatch(c["xq"], 3)
        assert E.GPP_ERR_ARG == again._lib.gpp_nipv_qbatch(again._h, 6, 3, E._ptr(np.ascontiguousarray(c["xq"])),
                                                            None, None, E._ptr(np.empty(6)), None, None)
    finally:
        again.close()


def test_argument_checks():
    from gpplus_b200 import _engine as E
    p = make_problem(100, 2, 0, seed=24)
    eng = _engine(p)
    try:
        eng.factorize(make_hyper(p, seed=1))
        x = np.ascontiguousarray(make_candidates(p, 129 * 2, seed=25)["xq"])
        for m, match in ((0, "GPP_MAX_IPV_POINTS"), (E.MAX_IPV_POINTS + 1, "GPP_MAX_IPV_POINTS")):
            rc = eng._lib.gpp_ipv_points(eng._h, m, E._ptr(x), None)
            assert rc == E.GPP_ERR_ARG and match.encode() in eng._lib.gpp_last_error()
        eng.ipv_points(x[:20])
        with pytest.raises(ValueError, match="GPP_MAX_QBATCH"):
            eng.nipv_qbatch(x, 129)
        vals = np.empty(2)
        for b, q, out, match in ((2, 0, vals, b"GPP_MAX_QBATCH"), (-1, 4, vals, b"b must be"),
                                 (2, 4, None, b"values missing")):
            rc = eng._lib.gpp_nipv_qbatch(eng._h, b, q, E._ptr(x), None, None, E._ptr(out), None, None)
            assert rc == E.GPP_ERR_ARG and match in eng._lib.gpp_last_error()
        v, d, jit = eng.nipv_qbatch(x[:0], 4)
        assert v.shape == (0,) and jit.shape == (0,)
    finally:
        eng.close()


def test_gradient_matches_central_differences():
    p = make_problem(200, 3, 2, dz=2, n_combo=3, n_noise=2, seed=21)
    h = make_hyper(p, seed=11, noise=1e-2)
    q, b = 4, 3
    c = make_candidates(p, b * q, seed=22)
    ipv = make_candidates(p, 300, seed=23)
    eng = _engine(p)
    try:
        eng.factorize(h)
        eng.ipv_points(ipv["xq"], level_idx=ipv["level_idx"])
        _, d, _ = eng.nipv_qbatch(c["xq"], q, **_kw(c))

        def f(x):
            return float(eng.nipv_qbatch(x, q, want_grad=False, **_kw(c))[0].sum())

        eps = 1e-6
        fd = np.zeros_like(d)
        for i in range(b * q):
            for k in range(p["dq"]):
                xp, xm = c["xq"].copy(), c["xq"].copy()
                xp[i, k] += eps
                xm[i, k] -= eps
                fd[i, k] = (f(xp) - f(xm)) / (2 * eps)
    finally:
        eng.close()
    print("d_xq vs central differences %.2e" % float(np.max(np.abs(d - fd))))
    np.testing.assert_allclose(d, fd, rtol=1e-5, atol=1e-7)


def _model(X, y):
    from gpplus_b200.models import GP_Plus
    return GP_Plus(torch.tensor(X), torch.tensor(y), dtype=torch.float64, quant_correlation_class="Matern52Kernel")


def test_model_end_to_end_and_the_optimizer_improves_on_screening():
    """-value is the mean latent predictive variance (no observation noise) at mc_points of the GP refitted on
    train + X_t with the same hyper-parameters (added y inside the training range, so the min-max scaling is
    unchanged)."""
    from gpplus_b200.bayesian_optimizations import optimize_acquisition_qbatch
    rng = np.random.default_rng(26)
    X = rng.uniform(-2, 2, (80, 3))
    y = np.sin(X[:, 0]) + 0.5 * np.cos(1.5 * X[:, 1]) + 0.2 * X[:, 2] + 0.02 * rng.standard_normal(80)
    m = _model(X, y)
    with torch.no_grad():
        m.covar_module.raw_outputscale.fill_(0.5)
        m.likelihood.noise_covar.raw_noise.fill_(-6.0)
    P = torch.tensor(rng.uniform(-2, 2, (500, 3)))
    b, q = 3, 4
    x0 = torch.tensor(rng.uniform(-2, 2, (b, q, 3)))
    xe = x0.clone().requires_grad_(True)
    val = m.acquisition_qbatch(xe, "qNIPV", mc_points=P)
    g, = torch.autograd.grad(val.sum(), xe)
    assert val.shape == (b,) and bool(torch.isfinite(g).all())
    for t in range(b):
        Xa = np.vstack([X, x0[t].numpy()])
        ya = np.concatenate([y, np.full(q, float(np.mean(y)))])
        m2 = _model(Xa, ya)
        assert float(m2.y_min) == float(m.y_min) and float(m2.y_std) == float(m.y_std)
        with torch.no_grad():
            for (n1, p1), (n2, p2) in zip(m.named_parameters(), m2.named_parameters()):
                assert n1 == n2
                p2.copy_(p1)
            _, sd = m2.predict(P, return_std=True, include_noise=False)
        want = -float((sd * sd).mean())
        got = float(val[t].detach())
        print("t-batch %d: nipv %.10e refit %.10e" % (t, got, want))
        assert abs(got - want) <= 1e-7 * abs(want)
        m2.release_engine()

    bounds = np.array([[-2.0] * 3, [2.0] * 3])
    Xopt, vopt = optimize_acquisition_qbatch(m, bounds, 4, "qNIPV", num_restarts=4, raw_samples=64,
                                             options={"maxiter": 40}, seed=7, mc_points=P)
    raw = torch.quasirandom.SobolEngine(dimension=12, scramble=True, seed=7).draw(64, dtype=torch.float64)
    with torch.no_grad():
        v_raw = m.acquisition_qbatch(-2.0 + 4.0 * raw.reshape(64, 4, 3), "qNIPV", mc_points=P)
    print("optimised qNIPV %.8e, best raw %.8e" % (vopt, float(v_raw.max())))
    assert Xopt.shape == (4, 3) and bool((Xopt.abs() <= 2.0).all())
    assert vopt > float(v_raw.max())
    m.release_engine()
