"""Parity pinned to the REFERENCE'S OWN CODE (SURVEY 8c).

``tests/golden/ref_*.npz`` are outputs of the unmodified files of a GP-Plus checkout, executed through the test-only
import shim ``oracle/_ref_shim`` by ``tests/golden/make_reference_fixtures.py``.  Here (CPU):

  * the CPU oracle (oracle/gpplus_oracle.py) is checked against those outputs -- this is what moves the oracle off
    "parity unpinned" for the rows GP+ itself owns (model construction, one-hot table, latent map, kernel tree,
    means, noise model, priors, MLLObjective packing);
  * the product's host-side logic (parameter / prior order, ``pack_parameters``, ``get_bounds``,
    ``_sample_from_prior``, priors, acquisition formulas, preprocessing, test functions) is checked against them;
  * when a GP-Plus checkout is present (``$GPPLUS_REFERENCE`` or ``oracle/_ref``; it is not part of this repository)
    the reference functions are additionally called LIVE on fresh random inputs.

The GPU half (engine vs the same fixtures through the C ABI) is tests/test_reference_pin_gpu.py.
"""
import glob
import json
import os
import warnings

import numpy as np
import pytest
import torch

from oracle import gpplus_oracle as GO

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
MODEL_CASES = sorted(os.path.basename(p)[4:-4] for p in glob.glob(os.path.join(GOLD, "ref_*.npz"))
                     if not p.endswith("ref_misc.npz"))

# tolerances against the all-float64 reference model ("f64" variant of the fixtures)
TOL_NLL = 1e-9      # relative, data term (north_star: 1e-9 on the MLL)
TOL_GRAD = 1e-8     # relative to the gradient's max-norm
# the priors of the reference hold float32 constants (gpytorch registers python-float prior parameters as float32
# buffers; .double() casts the rounded values), so the prior part of the posterior agrees to float32 epsilon only
TOL_POST = 2e-8


def post_scale(z, k):
    """Magnitude the posterior tolerance refers to: |data term| + |prior term| (their sum can cancel)."""
    nll, post = float(z["f_f64_nll"][k]), float(z["f_f64_post"][k])
    return abs(nll) + abs(post - nll)


def grad_tol(kw):
    """Gradient tolerance relative to the gradient's max-norm.  The probabilistic embedding of the reference copies
    the sampled latent positions into a float32 buffer (gp_plus.py:418, 435-436), so the gradient that flows back to
    the encoder weights is rounded to float32 there: its own gradient is float32-accurate only."""
    return 1e-6 if kw.get("embedding_type") == "probabilistic" else TOL_GRAD


def load_case(name):
    z = np.load(os.path.join(GOLD, "ref_%s.npz" % name))
    meta = json.loads(bytes(z["meta_json"]).decode())
    kw = dict(meta["kwargs"])
    if "qual_dict" in kw:
        kw["qual_dict"] = {int(k): int(v) for k, v in kw["qual_dict"].items()}
    return z, meta, kw


def oracle_spec(z, kw):
    spec = {"X": z["Xtr"], "y": z["ytr"], "qual_dict": kw.get("qual_dict", {}),
            "kernel": kw.get("quant_correlation_class", "Rough_RBF")}
    for k in ("multiple_noise", "m_gp", "m_gp_ref", "fix_noise", "fix_noise_val", "lb_noise", "interval_score",
              "embedding_type", "num_pass_train", "num_pass_pred", "seed_number"):
        if k in kw:
            spec[k] = kw[k]
    return spec


def build_product_model(z, kw):
    from gpplus_b200.models import GP_Plus
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return GP_Plus(torch.as_tensor(z["Xtr"]), torch.as_tensor(z["ytr"]), dtype=torch.float64, **kw)


def test_reference_fixtures_exist():
    assert len(MODEL_CASES) >= 9, MODEL_CASES
    assert os.path.exists(os.path.join(GOLD, "ref_misc.npz"))


@pytest.mark.parametrize("name", MODEL_CASES)
def test_oracle_matches_the_reference_objective(name):
    """oracle/gpplus_oracle.neg_log_posterior == reference MLLObjective.fun (float64 model), value and gradient."""
    z, meta, kw = load_case(name)
    spec = oracle_spec(z, kw)
    assert [n for n, _ in GO.theta_layout(spec)] == meta["param_names"]
    for k, th in enumerate(z["thetas"]):
        f, g = GO.neg_log_posterior(spec, th, add_prior=False)
        fr, gr = float(z["f_f64_nll"][k]), z["g_f64_nll"][k]
        assert abs(f - fr) <= TOL_NLL * abs(fr), (name, k, f, fr)
        assert np.max(np.abs(g - gr)) <= grad_tol(kw) * np.max(np.abs(gr)), (name, k)
        f, g = GO.neg_log_posterior(spec, th, add_prior=True)
        fr, gr = float(z["f_f64_post"][k]), z["g_f64_post"][k]
        assert abs(f - fr) <= TOL_POST * post_scale(z, k), (name, k, f, fr)
        assert np.max(np.abs(g - gr)) <= max(1e-7, grad_tol(kw)) * np.max(np.abs(gr)), (name, k)


@pytest.mark.parametrize("name", MODEL_CASES)
def test_reference_float32_residue_is_bounded(name):
    """The model exactly as the reference constructs it (dtype=torch.float64 but gpytorch's own parameters left in
    float32: noise transform and priors evaluated in float32) stays within float32 rounding of its float64 self;
    the FP64 engine targets the float64 variant."""
    z, _, _ = load_case(name)
    rel = np.abs(z["f_asbuilt_post"] - z["f_f64_post"]) / np.abs(z["f_f64_post"])
    assert rel.max() < 5e-5, rel
    gref = np.abs(z["g_f64_post"]).max(axis=1)
    assert (np.abs(z["g_asbuilt_post"] - z["g_f64_post"]).max(axis=1) / gref).max() < 5e-3


@pytest.mark.parametrize("name", MODEL_CASES)
def test_product_host_logic_matches_the_reference(name):
    """named_parameters / named_priors order, pack_parameters, get_bounds and the seeded prior draws."""
    from gpplus_b200.optim.mll_scipy import MLLObjective, _sample_from_prior, get_bounds
    z, meta, kw = load_case(name)
    m = build_product_model(z, kw)
    obj = MLLObjective(m, True, [0, 0])
    assert [n for n, p in m.named_parameters() if p.requires_grad] == meta["param_names"]
    assert [list(p.shape) for n, p in m.named_parameters() if p.requires_grad] == meta["param_shapes"]
    assert [n for n, *_ in m.named_priors()] == meta["prior_names"]
    theta0 = obj.pack_parameters()
    # everything but the randomly initialised latent map must start where the reference starts
    random_init = np.concatenate([np.full(int(np.prod(s)), n.startswith("latent") or n.startswith("A_matrix"))
                                  for n, s in zip(meta["param_names"], meta["param_shapes"])])
    np.testing.assert_allclose(theta0[~random_init], z["theta_init"][~random_init], rtol=0, atol=1e-7)
    lo, hi = get_bounds(obj, theta0)
    np.testing.assert_array_equal(lo, z["bounds_lo"])
    np.testing.assert_array_equal(hi, z["bounds_hi"])
    torch.manual_seed(7)
    draws = np.stack([_sample_from_prior(m) for _ in range(3)])
    # same torch RNG stream, same order of sampler calls -> the same starts as the reference's fit_model_scipy
    np.testing.assert_allclose(draws, z["prior_draws_seed7"], rtol=2e-6, atol=1e-7)


@pytest.mark.parametrize("name", MODEL_CASES)
def test_product_natural_parameters_reproduce_the_reference_through_the_oracle(name):
    """The raw -> natural transforms of the product model (what crosses the C ABI) fed to the natural-parameter
    oracle reproduce the reference's data term: pins GPR._natural / the latent table / index vectors on CPU."""
    from gpplus_b200.optim.mll_scipy import MLLObjective
    from oracle import gp_oracle as O
    z, meta, kw = load_case(name)
    if kw.get("interval_score"):
        pytest.skip("the interval-score penalty is not part of the data term")
    m = build_product_model(z, kw)
    obj = MLLObjective(m, False, [0, 0])
    x = m.train_inputs[0]
    cols = m._quant_columns()
    qk = m._quant_kernel() if len(cols) > 0 else None
    for k, th in enumerate(z["thetas"]):
        obj._load(th)
        with torch.no_grad():
            w, zt, sf2, noise, beta = m._natural()
        n_mean, _ = m._mean_layout()
        prob = {"n": x.shape[0], "dq": len(cols), "dz": 0 if zt.numel() == 0 else int(zt.shape[-1]),
                "n_combo": 0 if zt.numel() == 0 else int(zt.shape[-2]), "n_pass": int(zt.shape[0]) if zt.dim() == 3 else 1,
                "n_noise": int(noise.numel()), "n_mean": n_mean,
                "kernel": qk.family if qk is not None else 0, "xq": x[:, cols].double().numpy(),
                "y": m.train_targets.double().numpy(), "level_idx": m._level_index(x, True),
                "noise_idx": m._noise_index(x), "mean_idx": m._mean_index(x)}
        hyp = {"w": w.double().numpy(), "z": zt.double().numpy() if zt.numel() else None, "sigma_f2": float(sf2),
               "noise": noise.double().numpy(), "beta": beta.double().numpy() if n_mean > 0 else None}
        out = O.mll(prob, hyp, want_grad=False)
        fr = float(z["f_f64_nll"][k])
        assert abs(out["nll"] - fr) <= TOL_NLL * abs(fr), (name, k, out["nll"], fr)


def test_misc_helpers_match_the_reference_fixtures():
    from gpplus_b200.bayesian_optimizations import AFs
    from gpplus_b200.preprocessing import setlevels, standard
    from gpplus_b200.priors import LogHalfHorseshoePrior, MollifiedUniformPrior
    from gpplus_b200.test_functions.analytical import borehole, borehole_mixed_variables, wing
    from gpplus_b200.utils.interval_score import interval_score_function
    from gpplus_b200.utils.transforms import inv_softplus, softplus
    z = np.load(os.path.join(GOLD, "ref_misc.npz"))
    mean, std, xval = (torch.as_tensor(z[k]) for k in ("af_mean", "af_std", "af_xval"))
    cost = {str(i): float(c) for i, c in enumerate(z["af_cost"])}
    cost_fun = lambda x: cost[str(int(x))]  # noqa: E731
    for mx in (True, False):
        for bf in (48.5, -2.0):
            tag = "%s_%s" % ("max" if mx else "min", "pos" if bf > 0 else "neg")
            hf = AFs.AF_HF_Engineering(bf, mean.clone(), std.clone(), xval, cost_fun, maximize=mx, si=0.01)
            lf = AFs.AF_LF_Engineering(bf, mean.clone(), std.clone(), xval, cost_fun, maximize=mx, si=0.01)
            np.testing.assert_allclose(hf.numpy(), z["af_hf_" + tag], rtol=1e-12, atol=0)
            np.testing.assert_allclose(lf.numpy(), z["af_lf_" + tag], rtol=1e-12, atol=1e-300)
    a, b, c, d = standard(torch.as_tensor(z["std_X"]).clone(), {3: 4}, torch.as_tensor(z["std_Xt"]).clone())
    for got, key in ((a, "std_out_X"), (b, "std_out_Xt"), (c, "std_mean"), (d, "std_std")):
        np.testing.assert_allclose(np.asarray(got, dtype=np.float64), z[key], rtol=1e-13, atol=1e-15)
    np.testing.assert_array_equal(np.asarray(setlevels(torch.as_tensor(z["lv_in"].copy()), qual_index=[0, 2])),
                                  z["lv_out_cols02"])
    np.testing.assert_array_equal(np.asarray(setlevels(torch.as_tensor(z["lv_in"].copy()))), z["lv_out_all"])
    np.random.seed(123)  # "shuffle" resamples rows with numpy's global generator (analytical.py:38-41)
    np.testing.assert_allclose(np.asarray(wing(X=z["wing_X"].copy())), z["wing_y"], rtol=1e-13)
    np.random.seed(124)
    np.testing.assert_allclose(np.asarray(borehole(X=z["borehole_X"].copy())), z["borehole_y"], rtol=1e-13)
    for fn, kw, key in ((wing, dict(n=16, random_state=11), "wing_rs11"),
                        (borehole, dict(n=16, random_state=12), "borehole_rs12"),
                        (borehole_mixed_variables, dict(n=16, qual_dict={0: 5, 5: 5}, random_state=13), "bmv_rs13")):
        X, y = fn(**kw)
        np.testing.assert_allclose(np.asarray(X, dtype=np.float64), z[key + "_X"], rtol=1e-13, atol=1e-15)
        np.testing.assert_allclose(np.asarray(y, dtype=np.float64), z[key + "_y"], rtol=1e-13)
    v = torch.as_tensor(z["sp_in"])
    np.testing.assert_allclose(softplus(v).numpy(), z["sp_out"], rtol=1e-14)
    np.testing.assert_allclose(inv_softplus(softplus(v)).numpy(), z["isp_out"], rtol=1e-12, atol=1e-14)
    s, acc = interval_score_function(torch.as_tensor(z["is_Yu"]).clone(), torch.as_tensor(z["is_Yl"]).clone(),
                                     torch.as_tensor(z["is_Y"]))
    assert float(s) == pytest.approx(float(z["is_score"]), rel=1e-14)
    assert float(acc) == pytest.approx(float(z["is_acc"]), rel=1e-14)
    hs = LogHalfHorseshoePrior(0.01, 1e-8)
    np.testing.assert_allclose(hs.log_prob(torch.as_tensor(z["hs_x"])).numpy(), z["hs_logp"], rtol=2e-7, atol=2e-7)
    torch.manual_seed(5)
    np.testing.assert_allclose(hs.expand([4]).sample().double().numpy(), z["hs_sample_seed5"], rtol=2e-6)
    np.testing.assert_allclose(np.asarray(hs.expand([3]).lb, dtype=np.float64), z["hs_expand_lb"], rtol=1e-6)
    mu = MollifiedUniformPrior(np.log(0.1), np.log(10))
    np.testing.assert_allclose(mu.log_prob(torch.as_tensor(z["mu_x"])).numpy(), z["mu_logp"], rtol=2e-7, atol=2e-7)
    torch.manual_seed(6)
    np.testing.assert_allclose(mu.expand([5]).sample().double().numpy(), z["mu_sample_seed6"], rtol=2e-6)


# ------------------------------------------------------------------------------------------------
# live comparison with the reference (only where a GP-Plus checkout is present: GPPLUS_REFERENCE or oracle/_ref)
def _live():
    from oracle import _ref_shim
    if not _ref_shim.available():
        pytest.skip("no GP-Plus reference checkout to call live (set GPPLUS_REFERENCE or place one at oracle/_ref)")
    _ref_shim.install()


def test_live_reference_model_vs_oracle_on_fresh_data():
    """A model the fixtures do not contain: the reference's own objective, evaluated now, equals the oracle."""
    _live()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        from gpplus.models import GP_Plus as RefGP
        from gpplus.optim.mll_scipy import MLLObjective as RefObj
        rng = np.random.RandomState(21)
        n = 90
        X = np.hstack([rng.randint(0, 3, size=(n, 1)), rng.randn(n, 4), rng.randint(0, 2, size=(n, 1))]).astype(np.float64)
        y = np.sin(X[:, 1]) + 0.3 * X[:, 0] - 0.5 * X[:, 5] + 0.05 * rng.randn(n)
        qd = {0: 3, 5: 2}
        for kname in ("Rough_RBF", "Matern32Kernel", "Matern52Kernel", "RBFKernel"):
            m = RefGP(torch.as_tensor(X), torch.as_tensor(y), qual_dict=qd, dtype=torch.float64,
                      quant_correlation_class=kname, multiple_noise=True, m_gp="multiple_constant").double()
            obj = RefObj(m, True, [0, 0])
            th = (obj.pack_parameters() + 0.2 * rng.randn(obj.pack_parameters().size)).astype(np.float32).astype(np.float64)
            f, g = obj.fun(th.copy())
            spec = {"X": X, "y": y, "qual_dict": qd, "kernel": kname, "multiple_noise": True,
                    "m_gp": "multiple_constant"}
            fo, go = GO.neg_log_posterior(spec, th)
            assert abs(f - fo) <= TOL_POST * abs(fo), (kname, f, fo)
            assert np.max(np.abs(g - go)) <= 1e-7 * np.max(np.abs(go)), kname


def test_live_reference_helpers_on_random_inputs():
    _live()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        from gpplus.bayesian_optimizations import AFs as RAF
        from gpplus.preprocessing import setlevels as r_setlevels, standard as r_standard
        from gpplus.priors import LogHalfHorseshoePrior as RHS, MollifiedUniformPrior as RMU
        from gpplus.test_functions.analytical import borehole_mixed_variables as r_bmv, wing as r_wing
        from gpplus.utils.interval_score import interval_score_function as r_is
    from gpplus_b200.bayesian_optimizations import AFs
    from gpplus_b200.preprocessing import setlevels, standard
    from gpplus_b200.priors import LogHalfHorseshoePrior, MollifiedUniformPrior
    from gpplus_b200.test_functions.analytical import borehole_mixed_variables, wing
    from gpplus_b200.utils.interval_score import interval_score_function
    rng = np.random.RandomState(99)
    for trial in range(3):
        mean = torch.as_tensor(rng.randn(25, 1) * 2 + 3.0)
        std = torch.as_tensor(np.abs(rng.randn(25, 1)) + 0.05)
        xval = torch.as_tensor(np.hstack([rng.randn(25, 2), rng.randint(0, 2, size=(25, 1))]))
        cost_fun = lambda x: {0: 50.0, 1: 2.0}[int(x)]  # noqa: E731
        for mx in (True, False):
            a = RAF.AF_HF_Engineering(2.5, mean.clone(), std.clone(), xval, cost_fun, maximize=mx, si=0.0)
            b = AFs.AF_HF_Engineering(2.5, mean.clone(), std.clone(), xval, cost_fun, maximize=mx, si=0.0)
            np.testing.assert_allclose(b.numpy(), a.numpy(), rtol=1e-12)
            a = RAF.AF_LF_Engineering(2.5, mean.clone(), std.clone(), xval, cost_fun, maximize=mx, si=0.0)
            b = AFs.AF_LF_Engineering(2.5, mean.clone(), std.clone(), xval, cost_fun, maximize=mx, si=0.0)
            np.testing.assert_allclose(b.numpy(), a.numpy(), rtol=1e-12, atol=1e-300)
        X = torch.as_tensor(np.hstack([rng.randn(20, 2) * 5 + 1, rng.randint(0, 3, size=(20, 1))]))
        ra, rb, rc = r_standard(X.clone(), {2: 3})
        pa, pb, pc = standard(X.clone(), {2: 3})
        for u, v in ((ra, pa), (rb, pb), (rc, pc)):
            np.testing.assert_allclose(np.asarray(v, dtype=np.float64), np.asarray(u, dtype=np.float64), rtol=1e-13)
        raw = torch.as_tensor(rng.randint(0, 9, size=(12, 3)).astype(np.float64) * 1.5)
        np.testing.assert_array_equal(np.asarray(setlevels(raw.clone(), qual_index=[0, 1])),
                                      np.asarray(r_setlevels(raw.clone(), qual_index=[0, 1])))
        Xw = rng.rand(7, 10)
        np.random.seed(trial)
        mine = np.asarray(wing(X=Xw.copy()))
        np.random.seed(trial)
        np.testing.assert_allclose(mine, np.asarray(r_wing(X=Xw.copy())), rtol=1e-13)
        np.random.seed(50 + trial)  # the categorical levels come from numpy's global generator (analytical.py:121-125)
        Xa, ya = r_bmv(n=10, qual_dict={0: 5, 5: 5}, random_state=trial)
        np.random.seed(50 + trial)
        Xb, yb = borehole_mixed_variables(n=10, qual_dict={0: 5, 5: 5}, random_state=trial)
        np.testing.assert_allclose(np.asarray(Xb, dtype=np.float64), np.asarray(Xa, dtype=np.float64), rtol=1e-13)
        np.testing.assert_allclose(np.asarray(yb, dtype=np.float64), np.asarray(ya, dtype=np.float64), rtol=1e-13)
        Yu, Yl, Y = (torch.as_tensor(rng.randn(30) + s) for s in (1.0, -1.0, 0.0))
        assert float(interval_score_function(Yu.clone(), Yl.clone(), Y)[0]) == pytest.approx(
            float(r_is(Yu.clone(), Yl.clone(), Y)[0]), rel=1e-14)
        x = torch.as_tensor(rng.randn(9) * 3 - 4)
        np.testing.assert_allclose(LogHalfHorseshoePrior(0.01, 1e-8).log_prob(x).numpy(),
                                   RHS(0.01, 1e-8).log_prob(x).double().numpy(), rtol=2e-7, atol=2e-7)
        np.testing.assert_allclose(MollifiedUniformPrior(-2.3, 2.3).log_prob(x).numpy(),
                                   RMU(-2.3, 2.3).log_prob(x).double().numpy(), rtol=2e-7, atol=2e-7)
