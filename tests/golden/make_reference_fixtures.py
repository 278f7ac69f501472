"""Generate fixtures FROM THE REFERENCE ITSELF: a GP-Plus checkout's own, unmodified Python files are imported through
the test-only shim (oracle/_ref_shim: a fake ``gpplus`` package pointing at the checkout plus a dense-torch
re-statement of the gpytorch API the reference calls) and their outputs are stored next to this script.

    GPPLUS_REFERENCE=<GP-Plus checkout> python tests/golden/make_reference_fixtures.py   # ~1 min on CPU

What the fixtures pin (every number below is produced by the reference's code, not by this repo's):
  * model construction: parameter names / shapes / order (``named_parameters``), prior names / order
    (``named_priors``), ``MLLObjective.pack_parameters``, ``get_bounds``, ``_sample_from_prior`` (seeded);
  * ``MLLObjective.fun(theta)`` = negative log posterior and its autograd gradient, with and without priors,
    for the model as constructed with ``dtype=torch.float64`` (variant "asbuilt": gpytorch creates the noise,
    output-scale, lengthscale and mean parameters in float32, so the noise transform and the priors are evaluated
    in float32) and after ``model.double()`` (variant "f64": everything in float64 -- the parity target of the
    FP64 engine, tolerance 1e-9);
  * ``GP_Plus.predict`` (mean, std; with and without noise) on a mixed batch and on single-level batches;
  * host-side helpers: acquisition functions, ``standard``, ``setlevels``, analytical test functions, transforms,
    the interval score and the prior log-densities / samplers.

The gpytorch semantics underneath (kernel formulas, covar_dist, psd_safe_cholesky, ExactGP prediction) are the shim's
re-statement and remain unverifiable here; see oracle/_ref_shim/__init__.py.
"""
import json
import os
import sys
import warnings

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
warnings.filterwarnings("ignore")

from oracle import _ref_shim  # noqa: E402

_ref_shim.install()

from gpplus.bayesian_optimizations import AFs as RAF  # noqa: E402
from gpplus.models import GP_Plus  # noqa: E402
from gpplus.optim.mll_scipy import MLLObjective, _sample_from_prior, get_bounds  # noqa: E402
from gpplus.preprocessing import setlevels, standard, train_test_split_normalizeX  # noqa: E402
from gpplus.priors import LogHalfHorseshoePrior, MollifiedUniformPrior  # noqa: E402
from gpplus.test_functions.analytical import borehole, borehole_mixed_variables, wing  # noqa: E402
from gpplus.test_functions.multi_fidelity import Borehole_MF_BO, multi_fidelity_wing  # noqa: E402
from gpplus.utils import set_seed  # noqa: E402
from gpplus.utils.interval_score import interval_score_function  # noqa: E402
from gpplus.utils.transforms import inv_softplus, softplus  # noqa: E402


def _np(t):
    return t.detach().cpu().double().numpy() if torch.is_tensor(t) else np.asarray(t, dtype=np.float64)


def model_case(name, Xtr, ytr, Xte, kwargs, single_level_col=None):
    """Run the reference model on one data set and store everything a parity test needs."""
    Xtr, ytr, Xte = torch.as_tensor(_np(Xtr)), torch.as_tensor(_np(ytr)).reshape(-1), torch.as_tensor(_np(Xte))
    blob = {"Xtr": _np(Xtr), "ytr": _np(ytr), "Xte": _np(Xte)}
    meta = {"kwargs": {k: (v if not isinstance(v, dict) else {str(a): int(b) for a, b in v.items()})
                       for k, v in kwargs.items()}}

    def build(double):
        set_seed(1)
        m = GP_Plus(Xtr.clone(), ytr.clone(), dtype=torch.float64, **kwargs)
        return m.double() if double else m

    m64 = build(True)
    obj = MLLObjective(m64, True, [0, 0])
    meta["param_names"] = [n for n, p in m64.named_parameters() if p.requires_grad]
    meta["param_shapes"] = [list(p.shape) for n, p in m64.named_parameters() if p.requires_grad]
    meta["all_param_names"] = [n for n, p in m64.named_parameters()]
    meta["prior_names"] = [n for n, *_ in m64.named_priors()]
    theta_init = obj.pack_parameters().astype(np.float64)
    torch.manual_seed(7)
    draws = [_sample_from_prior(m64).astype(np.float64) for _ in range(3)]
    blob["prior_draws_seed7"] = np.stack(draws)
    lo, hi = get_bounds(obj, theta_init)
    blob["bounds_lo"], blob["bounds_hi"] = np.asarray(lo, dtype=np.float64), np.asarray(hi, dtype=np.float64)
    blob["theta_init"] = theta_init
    # evaluation points: a shifted theta_init and two prior draws pulled towards moderate conditioning
    rng = np.random.RandomState(3)
    thetas = [theta_init + 0.1, 0.5 * draws[0] + 0.05 * rng.randn(theta_init.size), 0.3 * draws[1]]
    thetas = [np.asarray(t, dtype=np.float32).astype(np.float64) for t in thetas]  # what fun() sees after its cast
    blob["thetas"] = np.stack(thetas)
    for variant, double in (("f64", True), ("asbuilt", False)):
        for add_prior in (True, False):
            fs, gs = [], []
            for th in thetas:
                m = build(double)
                f, g = MLLObjective(m, add_prior, [0, 0]).fun(th.copy())
                fs.append(f)
                gs.append(np.asarray(g, dtype=np.float64))
            key = "%s_%s" % (variant, "post" if add_prior else "nll")
            blob["f_" + key], blob["g_" + key] = np.asarray(fs), np.stack(gs)
    # predictions at thetas[0] (float64 model)
    m = build(True)
    o = MLLObjective(m, True, [0, 0])
    o.fun(thetas[0].copy())  # loads theta into the model
    for inc in (True, False):
        mu, sd = m.predict(Xte.clone(), return_std=True, include_noise=inc)
        tag = "noise" if inc else "nonoise"
        blob["pred_mean_" + tag], blob["pred_std_" + tag] = _np(mu), _np(sd)
    if single_level_col is not None:
        # batches that hold ONE level of a categorical column: eval-mode setlevels ranks [train, test] together
        lv = np.unique(_np(Xte)[:, single_level_col])
        blob["single_levels"] = lv
        for k, v in enumerate(lv):
            rows = Xte[Xte[:, single_level_col] == v]
            mu, sd = m.predict(rows.clone(), return_std=True, include_noise=True)
            blob["single_%d_mean" % k], blob["single_%d_std" % k] = _np(mu), _np(sd)
        mu, sd = m.predict(Xte[:1].clone(), return_std=True, include_noise=True)
        blob["one_row_mean"], blob["one_row_std"] = _np(mu), _np(sd)
    if "qual_dict" not in kwargs and not kwargs.get("interval_score"):
        # Adam path (optim/mll_torch.py:56-141): loss history of 6 steps from thetas[0]; the loss is
        # -(log p(y) + log priors) / n (gpytorch ExactMarginalLogLikelihood)
        from gpplus.optim.mll_torch import fit_model_torch
        m = build(True)
        MLLObjective(m, True, [0, 0]).fun(thetas[0].copy())
        f_inc, hist = fit_model_torch(m, num_iter=6, num_restarts=0, lr_default=0.01)
        blob["adam_loss_hist"] = np.asarray(hist[0], dtype=np.float64)
        blob["adam_f_inc"] = np.asarray(f_inc, dtype=np.float64)
        blob["adam_theta_end"] = MLLObjective(m, True, [0, 0]).pack_parameters().astype(np.float64)
    blob["meta_json"] = np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8)
    np.savez_compressed(os.path.join(HERE, "ref_%s.npz" % name), **blob)
    print("ref_%s: n=%d p=%d f64 posterior %s" % (name, Xtr.shape[0], theta_init.size, blob["f_f64_post"]), flush=True)


def main_models():
    # C1: borehole emulation (Example 01), rough-RBF, no categorical input
    set_seed(4)
    X, y = borehole(n=800, random_state=4)
    Xtr, Xte, ytr, yte = train_test_split_normalizeX(X, y, test_size=0.75, qual_dict={})
    model_case("c1_borehole_rough", Xtr, ytr, Xte[:48], {})
    # the other quantitative kernels on the same data
    for kname in ("RBFKernel", "Matern32Kernel", "Matern52Kernel"):
        model_case("c1_borehole_" + kname.lower(), Xtr[:120], ytr[:120], Xte[:32], {"quant_correlation_class": kname})
    # C2: mixed-variable borehole (Example 02): two categorical inputs x 5 levels, 2-D latent map
    set_seed(4)
    qd = {0: 5, 5: 5}
    X, y = borehole_mixed_variables(n=1200, qual_dict=qd, random_state=4)
    Xtr, Xte, ytr, yte = train_test_split_normalizeX(X, y, test_size=0.75, qual_dict=qd)
    model_case("c2_mixed_rough", Xtr, ytr, Xte[:64], {"qual_dict": qd}, single_level_col=0)
    # probabilistic embedding (variational encoder, seeded epsilon) with one and with three forward passes: the
    # multi-pass ensemble covariance Sigma = (1/k) sum_p (K_p + m m^T) - m m^T (gp_plus.py:387-399, 414-461, 474-482)
    model_case("c2_mixed_probabilistic_p1", Xtr[:150], ytr[:150], Xte[:32],
               {"qual_dict": qd, "embedding_type": "probabilistic"}, single_level_col=0)
    model_case("c2_mixed_probabilistic_p3", Xtr[:150], ytr[:150], Xte[:32],
               {"qual_dict": qd, "embedding_type": "probabilistic", "num_pass_train": 3, "num_pass_pred": 3,
                "quant_correlation_class": "Matern52Kernel"}, single_level_col=0)
    # C3: multi-fidelity wing (Example 03): 4 sources, one noise per source, one mean per source
    set_seed(4)
    X, y = multi_fidelity_wing(n={"0": 50, "1": 100, "2": 100, "3": 100},
                               noise_std={"0": 0.5, "1": 1.0, "2": 1.5, "3": 2.0}, random_state=4)
    qd = {10: 4}
    Xtr, Xte, ytr, yte = train_test_split_normalizeX(X, y, test_size=0.5, qual_dict=qd,
                                                     stratify=X[..., list(qd.keys())])
    Xtr3, ytr3, Xte3 = Xtr, ytr, Xte
    model_case("c3_wing_mf", Xtr, ytr, Xte[:64], {"qual_dict": qd, "multiple_noise": True, "m_gp": "multiple_constant"},
               single_level_col=10)
    model_case("c3_wing_mf_constref", Xtr[:90], ytr[:90], Xte[:32],
               {"qual_dict": qd, "multiple_noise": True, "m_gp": "multiple_constant", "m_gp_ref": "constant"},
               single_level_col=10)
    # C4 (small): wing, Matern-5/2, single constant mean -- the headline model at a size the CPU handles
    set_seed(4)
    X, y = wing(n=600, noise_std=0.5, random_state=4)
    Xtr, Xte, ytr, yte = train_test_split_normalizeX(X, y, test_size=0.5, qual_dict={})
    model_case("c4_wing_matern52", Xtr, ytr, Xte[:48], {"quant_correlation_class": "Matern52Kernel"})
    # C5: MFBO borehole (Example 04): 8 quantitative inputs + source (5 levels), one noise, zero / fixed-noise variants
    np.random.seed(0)
    U, y = Borehole_MF_BO(True, {"0": 5, "1": 5, "2": 50, "3": 5, "4": 50})
    qd = {8: 5}
    U, umean, ustd = standard(torch.tensor(U), qd)
    rng = np.random.RandomState(5)
    Xte = torch.cat([torch.as_tensor(rng.randn(60, 8)), torch.as_tensor(rng.randint(0, 5, size=(60, 1)), dtype=torch.float64)], 1)
    model_case("c5_mfbo_borehole", U, torch.tensor(y).reshape(-1), Xte, {"qual_dict": qd}, single_level_col=8)
    model_case("c5_mfbo_fixnoise_zero", U, torch.tensor(y).reshape(-1), Xte[:16],
               {"qual_dict": qd, "fix_noise": True, "fix_noise_val": 1e-4, "m_gp": "single_zero"})
    # interval-score penalty of the BO loop (mll_scipy.py:57-59; BO() builds its models with IS=True)
    model_case("c5_mfbo_interval_score", U, torch.tensor(y).reshape(-1), Xte[:16],
               {"qual_dict": qd, "interval_score": True})
    model_case("c3_wing_mf_interval_score", Xtr3[:90], ytr3[:90], Xte3[:16],
               {"qual_dict": {10: 4}, "multiple_noise": True, "m_gp": "multiple_constant", "interval_score": True})


def main_misc():
    """Host-side helpers: outputs of the reference functions on fixed inputs."""
    blob = {}
    rng = np.random.RandomState(0)
    # acquisition functions (AFs.py:102-159) -- x_val's last column is the source, cost by source
    mean = torch.as_tensor(rng.randn(40, 1) * 3.0 + 50.0)
    std = torch.as_tensor(np.abs(rng.randn(40, 1)) + 0.1)
    xval = torch.as_tensor(np.hstack([rng.randn(40, 3), rng.randint(0, 3, size=(40, 1))]))
    cost = {"0": 1000.0, "1": 100.0, "2": 10.0}
    cost_fun = lambda x: cost[str(int(x))]  # noqa: E731
    blob["af_mean"], blob["af_std"], blob["af_xval"] = _np(mean), _np(std), _np(xval)
    blob["af_cost"] = np.array([1000.0, 100.0, 10.0])
    for mx in (True, False):
        for bf in (48.5, -2.0):
            tag = "%s_%s" % ("max" if mx else "min", "pos" if bf > 0 else "neg")
            blob["af_hf_" + tag] = _np(RAF.AF_HF_Engineering(bf, mean.clone(), std.clone(), xval, cost_fun, maximize=mx, si=0.01))
            blob["af_lf_" + tag] = _np(RAF.AF_LF_Engineering(bf, mean.clone(), std.clone(), xval, cost_fun, maximize=mx, si=0.01))
    # preprocessing
    X = torch.as_tensor(np.hstack([rng.randn(30, 3) * [1.0, 10.0, 0.1] + [0.0, 5.0, -2.0], rng.randint(0, 4, size=(30, 1))]))
    Xt = torch.as_tensor(np.hstack([rng.randn(9, 3), rng.randint(0, 4, size=(9, 1))]))
    blob["std_X"], blob["std_Xt"] = _np(X), _np(Xt)
    a, b, c, d = standard(X.clone(), {3: 4}, Xt.clone())
    blob["std_out_X"], blob["std_out_Xt"], blob["std_mean"], blob["std_std"] = _np(a), _np(b), _np(c), _np(d)
    raw = np.array([[3.5, 1.0, 7.0], [1.5, 1.0, 9.0], [3.5, 2.0, 7.0], [2.5, 4.0, 8.0]])
    blob["lv_in"] = raw
    blob["lv_out_cols02"] = _np(setlevels(torch.as_tensor(raw.copy()), qual_index=[0, 2]))
    blob["lv_out_all"] = _np(setlevels(torch.as_tensor(raw.copy())))
    # analytical functions with explicit inputs
    Xw = rng.rand(20, 10)
    blob["wing_X"] = Xw
    np.random.seed(123)  # "shuffle" resamples rows with numpy's global generator (analytical.py:38-41)
    blob["wing_y"] = _np(wing(X=Xw.copy()))
    Xb = rng.rand(20, 8)
    blob["borehole_X"] = Xb
    np.random.seed(124)
    blob["borehole_y"] = _np(borehole(X=Xb.copy()))
    Xs, ys = wing(n=16, random_state=11)
    blob["wing_rs11_X"], blob["wing_rs11_y"] = _np(Xs), _np(ys)
    Xs, ys = borehole(n=16, random_state=12)
    blob["borehole_rs12_X"], blob["borehole_rs12_y"] = _np(Xs), _np(ys)
    Xs, ys = borehole_mixed_variables(n=16, qual_dict={0: 5, 5: 5}, random_state=13)
    blob["bmv_rs13_X"], blob["bmv_rs13_y"] = _np(Xs), _np(ys)
    # transforms, interval score
    v = torch.as_tensor(np.linspace(-8.0, 8.0, 33))
    blob["sp_in"], blob["sp_out"] = _np(v), _np(softplus(v))
    blob["isp_out"] = _np(inv_softplus(softplus(v)))
    Yu, Yl, Y = torch.as_tensor(rng.randn(50) + 1.0), torch.as_tensor(rng.randn(50) - 1.0), torch.as_tensor(rng.randn(50) * 2)
    s, acc = interval_score_function(Yu.clone(), Yl.clone(), Y)
    blob["is_Yu"], blob["is_Yl"], blob["is_Y"], blob["is_score"], blob["is_acc"] = _np(Yu), _np(Yl), _np(Y), _np(s), _np(acc)
    # priors: log-densities (float64 arguments) and seeded samples
    x = torch.as_tensor(np.linspace(-12.0, 3.0, 31))
    hs = LogHalfHorseshoePrior(0.01, 1e-8)
    blob["hs_x"], blob["hs_logp"] = _np(x), _np(hs.log_prob(x))
    torch.manual_seed(5)
    blob["hs_sample_seed5"] = _np(hs.expand([4]).sample())
    blob["hs_expand_lb"] = _np(hs.expand([3]).lb)
    mu_ = MollifiedUniformPrior(np.log(0.1), np.log(10))
    xm = torch.as_tensor(np.linspace(-4.0, 4.0, 33))
    blob["mu_x"], blob["mu_logp"] = _np(xm), _np(mu_.log_prob(xm))
    torch.manual_seed(6)
    blob["mu_sample_seed6"] = _np(mu_.expand([5]).sample())
    np.savez_compressed(os.path.join(HERE, "ref_misc.npz"), **blob)
    print("ref_misc: %d arrays" % len(blob), flush=True)


if __name__ == "__main__":
    main_misc()
    main_models()
