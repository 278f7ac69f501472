"""Parity of the CUDA path (through the C ABI) against the CPU oracle on seeded inputs.

Tolerances (FP64): |d nll| <= 1e-9 |nll| (BASELINE.json north_star), K entries 1e-12 relative to max|K|,
gradients 1e-8 relative to the largest gradient entry, predictions 1e-9.
"""
import glob
import os

import numpy as np
import pytest

from problems import engine_kwargs, make_candidates, make_hyper, make_problem

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))

NLL_RTOL = 1e-9
GRAD_RTOL = 1e-8
PRED_TOL = 1e-9


def rel(a, b):
    a, b = np.asarray(a, dtype=float), np.asarray(b, dtype=float)
    return float(np.max(np.abs(a - b)) / max(1e-300, np.max(np.abs(b))))


def check_case(p, h, mode="expansion", cand=48):
    from gpplus_b200 import _engine as E
    from oracle import gp_oracle as O
    ref = O.mll(p, h, want_grad=True, mode=mode, return_mats=True)
    eng = E.Engine(**engine_kwargs(p))
    try:
        assert rel(eng.covariance(h), ref["K"]) < 1e-12
        out = eng.mll_grad(h, want_grad=True)
        assert abs(out["nll"] - ref["nll"]) <= NLL_RTOL * abs(ref["nll"])
        assert out["jitter"] == ref["jitter"]
        for k in ("d_w", "d_noise", "d_z", "d_beta"):
            if k in ref and np.size(ref[k]):
                assert rel(out[k], ref[k]) < GRAD_RTOL, k
        assert abs(out["d_sigma_f2"] - ref["d_sigma_f2"]) <= GRAD_RTOL * max(1.0, abs(ref["d_sigma_f2"]))
        val = eng.mll_grad(h, want_grad=False)
        assert val["nll"] == out["nll"]  # value-only path is bit-identical to the value of the gradient path
        c = make_candidates(p, cand)
        for inc in (False, True):
            mu_ref, var_ref = O.predict(p, h, c, include_noise=inc, mode=mode)
            mu, var = eng.predict(c["xq"], c["level_idx"], c["noise_idx"], c["mean_idx"], include_noise=inc)
            assert np.max(np.abs(mu - mu_ref)) < PRED_TOL * max(1.0, np.max(np.abs(mu_ref)))
            assert np.max(np.abs(var - var_ref)) < PRED_TOL * max(1.0, np.max(np.abs(var_ref)))
    finally:
        eng.close()


@pytest.mark.parametrize("kind", [0, 1, 2])
@pytest.mark.parametrize("n", [1, 2, 127, 128, 129, 300])
def test_quantitative_kernels(kind, n):
    p = make_problem(n, 5, kind, seed=100 + n)
    check_case(p, make_hyper(p, seed=n))


@pytest.mark.parametrize("kind", [0, 2])
def test_latent_map_multi_noise_multi_mean(kind):
    p = make_problem(420, 10, kind, dz=2, n_combo=25, n_noise=4, n_mean=4, seed=21, zero_mean_group=True)
    check_case(p, make_hyper(p, seed=5))


def test_latent_only_no_quantitative_inputs():
    p = make_problem(150, 0, 0, dz=2, n_combo=12, seed=22)
    check_case(p, make_hyper(p, seed=6, noise=1e-2))


def test_wide_inputs_and_4d_latent():
    p = make_problem(260, 32, 1, dz=4, n_combo=7, seed=23)
    check_case(p, make_hyper(p, seed=7, w_scale=0.05))


def test_zero_mean_and_direct_distance_oracle():
    p = make_problem(200, 3, 2, n_mean=0, seed=24)
    check_case(p, make_hyper(p, seed=8), mode="direct")


def test_nine_tiles_recursive_inverse_non_power_of_two():
    p = make_problem(1100, 10, 2, seed=25)
    check_case(p, make_hyper(p, seed=9))


def test_factor_solves_and_inverse_identities_n2048():
    """Size-independent properties at a size the oracle is not asked to factor: L L^T = K_y, L^-1 L = I,
    K_y alpha = r, K_y^-1 symmetric."""
    from gpplus_b200 import _engine as E
    p = make_problem(2048, 10, 2, seed=26)
    h = make_hyper(p, seed=10)
    eng = E.Engine(**engine_kwargs(p))
    try:
        K = eng.covariance(h)
        assert np.array_equal(K, K.T)
        eng.mll_grad(h, want_grad=True)
        Ky = K + h["noise"][0] * np.eye(p["n"])
        L, Li, Ki, al = eng.fetch("L"), eng.fetch("Linv"), eng.fetch("Kinv"), eng.fetch("alpha")
        assert np.max(np.abs(L @ L.T - Ky)) < 1e-12
        assert np.max(np.abs(Li @ L - np.eye(p["n"]))) < 1e-9
        assert np.array_equal(Ki, Ki.T)
        assert np.max(np.abs(Ki @ Ky - np.eye(p["n"]))) < 1e-7
        r = p["y"] - h["beta"][0]
        assert np.max(np.abs(Ky @ al - r)) < 1e-9
    finally:
        eng.close()


def test_jitter_ladder_and_error_mapping():
    from gpplus_b200 import _engine as E
    from oracle import gp_oracle as O
    p = make_problem(64, 2, 0, seed=27)
    p["xq"][1] = p["xq"][0]  # duplicated point: K has a zero eigenvalue
    h = make_hyper(p, seed=11)
    # natural-parameter ABI: a slightly negative diagonal term makes K_y indefinite by a margin far above
    # rounding (lambda_min = -5e-9), so the outcome of the first rung does not depend on the rounding of the
    # factorisation; the 1e-8 rung of psd_safe_cholesky repairs it (lambda_min = +5e-9)
    h["noise"] = np.array([-5e-9])
    eng = E.Engine(**engine_kwargs(p))
    try:
        try:
            ref = O.mll(p, h, want_grad=False)
            out = eng.mll_grad(h, want_grad=True)
            assert out["jitter"] == ref["jitter"] and out["jitter"] > 0
            assert abs(out["nll"] - ref["nll"]) <= 1e-6 * abs(ref["nll"])  # kappa ~ 1e8 here
        except O.NotPSDError:
            with pytest.raises(E.NotPSDError):
                eng.mll_grad(h, want_grad=True)
        hn = dict(h)
        hn["sigma_f2"] = -1.0  # indefinite: every rung of the ladder fails
        with pytest.raises(E.NotPSDError):
            eng.mll_grad(hn, want_grad=True)
        hn["sigma_f2"] = float("nan")
        with pytest.raises(E.NanError):
            eng.mll_grad(hn, want_grad=True)
        out = eng.mll_grad(make_hyper(p, seed=12, noise=1e-2), want_grad=True)  # the handle survives failures
        assert np.isfinite(out["nll"])
    finally:
        eng.close()


def test_acquisition_argmax_matches_oracle():
    from gpplus_b200 import _engine as E
    from oracle import gp_oracle as O
    p = make_problem(180, 8, 0, dz=2, n_combo=5, n_noise=5, n_mean=1, seed=28)
    h = make_hyper(p, seed=13)
    c = make_candidates(p, 5000, seed=3)
    src = c["level_idx"].astype(np.int32)
    cost = np.array([1000.0, 100.0, 10.0, 100.0, 10.0])
    kinds = [E.ACQ_HF, E.ACQ_LF, E.ACQ_LF, E.ACQ_LF, E.ACQ_EI]
    best_f = np.array([0.4, 0.5, 0.6, 0.5, 0.45])
    eng = E.Engine(**engine_kwargs(p))
    try:
        eng.factorize(h)
        for maximize in (True, False):
            s, i, scores = eng.acq_argmax(c["xq"], src, cost, kinds, best_f, level_idx=c["level_idx"],
                                          maximize=maximize, y_min=2.0, y_std=3.0, return_scores=True)
            mu, var = O.predict(p, h, c, include_noise=False)
            mean, std = 2.0 + 3.0 * mu, np.sqrt(var) * 3.0
            want = np.empty(c["m"])
            for k in range(5):
                sel = src == k
                want[sel] = O.acquisition(mean[sel], std[sel], kinds[k], best_f[k], cost[k] * np.ones(sel.sum()),
                                          maximize=maximize)
            assert np.max(np.abs(scores - want)) < 1e-9 * max(1.0, np.max(np.abs(want)))
            assert i == int(np.argmax(want)) and s == scores[i]
    finally:
        eng.close()


def test_prediction_chunking_is_invisible():
    """A candidate table larger than one device chunk gives the same numbers as small calls."""
    from gpplus_b200 import _engine as E
    p = make_problem(16500, 4, 0, seed=29)  # np = 16512 -> chunk of 8064 candidates
    h = make_hyper(p, seed=14, noise=1e-2)
    c = make_candidates(p, 9000, seed=4)
    eng = E.Engine(**engine_kwargs(p))
    try:
        eng.factorize(h)
        mu, var = eng.predict(c["xq"])
        mu2, var2 = eng.predict(c["xq"][8000:8100])
        assert np.array_equal(mu[8000:8100], mu2) and np.array_equal(var[8000:8100], var2)
        assert np.all(var >= 1e-10) and np.all(np.isfinite(mu))
    finally:
        eng.close()


def test_golden_fixtures():
    from gpplus_b200 import _engine as E
    files = sorted(f for f in glob.glob(os.path.join(HERE, "golden", "*.npz")) if not os.path.basename(f).startswith("ref_"))
    assert len(files) >= 6
    for f in files:
        g = np.load(f)
        p = {k[2:]: g[k] for k in g.files if k.startswith("p_")}
        for k in ("n", "dq", "dz", "n_combo", "n_noise", "n_mean", "kernel"):
            p[k] = int(p[k])
        for k in ("level_idx", "noise_idx", "mean_idx"):
            p.setdefault(k, None)
        h = {k[2:]: g[k] for k in g.files if k.startswith("h_")}
        h["sigma_f2"] = float(h["sigma_f2"])
        h.setdefault("z", None)
        h.setdefault("beta", None)
        c = {k[2:]: g[k] for k in g.files if k.startswith("c_")}
        eng = E.Engine(**engine_kwargs(p))
        try:
            out = eng.mll_grad(h, want_grad=True)
            assert abs(out["nll"] - float(g["r_nll"])) <= NLL_RTOL * abs(float(g["r_nll"])), f
            assert rel(out["d_w"], g["r_d_w"]) < GRAD_RTOL, f
            assert rel(out["d_noise"], g["r_d_noise"]) < GRAD_RTOL, f
            if "r_d_z" in g.files:
                assert rel(out["d_z"], g["r_d_z"]) < GRAD_RTOL, f
            mu, var = eng.predict(c["xq"], c.get("level_idx"), c.get("noise_idx"), c.get("mean_idx"),
                                  include_noise=True)
            assert np.max(np.abs(mu - g["r_pred_mean"])) < PRED_TOL, f
            assert np.max(np.abs(var - g["r_pred_var"])) < PRED_TOL, f
        finally:
            eng.close()


def test_bitwise_reproducible_and_thread_safe_across_handles():
    import threading
    from gpplus_b200 import _engine as E
    p = make_problem(700, 6, 2, dz=2, n_combo=9, seed=30)
    h = make_hyper(p, seed=15)
    base = E.Engine(**engine_kwargs(p))
    ref = base.mll_grad(h)
    again = base.mll_grad(h)
    assert ref["nll"] == again["nll"] and np.array_equal(ref["d_w"], again["d_w"])
    base.close()
    results = [None] * 4

    def work(k):
        e = E.Engine(**engine_kwargs(p))
        for _ in range(3):
            results[k] = e.mll_grad(h)
        e.close()

    ts = [threading.Thread(target=work, args=(k,)) for k in range(4)]
    [t.start() for t in ts]
    [t.join() for t in ts]
    for r in results:
        assert r["nll"] == ref["nll"] and np.array_equal(r["d_z"], ref["d_z"])


@pytest.mark.parametrize("n", [513, 700, 1100, 1537, 2300])
def test_schedule_variants_are_bitwise_identical(n, monkeypatch):
    """The overlapped inverse (third stream), the CUDA-graph replay and the plain blocked factorisation are
    schedules of the same tile computations: L^-1, K^-1, the likelihood and its gradient must not change by a bit."""
    from gpplus_b200 import _engine as E
    p = make_problem(n, 5, 2, dz=2, n_combo=7, n_noise=2, seed=31)
    h = make_hyper(p, seed=13)
    results, launches = [], []
    # every configuration gets a handle built under its own settings: a parked handle of the same shape is only
    # handed back under the configuration it was created with (gpp_create compares them)
    for env in ({"GPP_OVERLAP_INV": "1", "GPP_GRAPH": "1"}, {"GPP_OVERLAP_INV": "0", "GPP_GRAPH": "0"},
                {"GPP_OVERLAP_INV": "1", "GPP_GRAPH": "0"}, {"GPP_CHOL": "blocked", "GPP_GRAPH": "0"}):
        for k in ("GPP_OVERLAP_INV", "GPP_GRAPH", "GPP_CHOL"):
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        eng = E.Engine(**engine_kwargs(p))
        try:
            assert eng.fp64_mode() == E.FP64_DMMA
            out = eng.mll_grad(h, want_grad=True)
            before = E.launch_count()
            out2 = eng.mll_grad(h, want_grad=True)  # second call replays the captured graph
            launches.append(E.launch_count() - before)
            assert out["nll"] == out2["nll"] and np.array_equal(out["d_w"], out2["d_w"])
            results.append((out, eng.fetch("Linv"), eng.fetch("Kinv")))
        finally:
            eng.close()
    # the blocked factorisation is a different chain of launches than the look-ahead schedule (same GPP_GRAPH=0);
    # at T = 5 (n = 513) both happen to issue 29 launches per evaluation
    if n > 640:
        assert launches[3] != launches[2], launches
    ref = results[0]
    for out, li, ki in results[1:3]:
        assert out["nll"] == ref[0]["nll"]
        assert np.array_equal(out["d_w"], ref[0]["d_w"]) and np.array_equal(out["d_z"], ref[0]["d_z"])
        assert np.array_equal(li, ref[1]) and np.array_equal(ki, ref[2])
    # the blocked driver groups the trailing updates differently (K = 512 panels): same result up to rounding
    out, li, ki = results[3]
    assert abs(out["nll"] - ref[0]["nll"]) <= 1e-11 * abs(ref[0]["nll"])
    assert np.max(np.abs(ki - ref[2])) <= 1e-9 * np.max(np.abs(ref[2]))


def test_recycled_handles_give_the_results_of_fresh_ones():
    """gpp_destroy parks small handles, gpp_create hands them back for a problem of the same shape: the recycled
    handle (captured CUDA graphs included) must evaluate the NEW training set, bit for bit like a fresh handle."""
    from gpplus_b200 import _engine as E
    E.pool_clear()
    pa = make_problem(n=300, dq=5, kernel=2, dz=2, n_combo=6, n_noise=2, n_mean=2, seed=41)
    pb = make_problem(n=300, dq=5, kernel=2, dz=2, n_combo=6, n_noise=2, n_mean=2, seed=42)
    ha, hb = make_hyper(pa, seed=43), make_hyper(pb, seed=44)
    fresh_b = E.Engine(**engine_kwargs(pb))
    want = fresh_b.mll_grad(hb, want_grad=True)
    cand = make_candidates(pb, 40, seed=45)
    fresh_b.factorize(hb)
    mu_w, var_w = fresh_b.predict(cand["xq"], level_idx=cand["level_idx"], noise_idx=cand["noise_idx"],
                                  mean_idx=cand["mean_idx"], include_noise=True)
    first = E.Engine(**engine_kwargs(pa))
    first.mll_grad(ha, want_grad=True)   # captures the graphs on problem A
    first.mll_grad(ha, want_grad=False)
    first.close()                        # parked
    again = E.Engine(**engine_kwargs(pb))  # recycled: same shape, new data
    got = again.mll_grad(hb, want_grad=True)
    assert got["nll"] == want["nll"]
    for k in ("d_w", "d_z", "d_noise", "d_beta"):
        assert np.array_equal(got[k], want[k]), k
    again.factorize(hb)
    mu, var = again.predict(cand["xq"], level_idx=cand["level_idx"], noise_idx=cand["noise_idx"],
                            mean_idx=cand["mean_idx"], include_noise=True)
    assert np.array_equal(mu, mu_w) and np.array_equal(var, var_w)
    assert again.stats()["evaluations"] == 2  # counters restart with the new problem
    again.close()
    fresh_b.close()
    E.pool_clear()


def test_pooled_handles_follow_the_settings_in_force(monkeypatch):
    """A handle parked under one configuration is not handed back under another: set_fp64_mode ("for engines created
    afterwards") and the per-handle switches read by gpp_create apply to the next create of the same shape, in both
    orders.  N = 1100 (T = 9) is pooled and small enough for the forced INT8-sliced arithmetic (T >= 8)."""
    from gpplus_b200 import _engine as E
    p = make_problem(1100, 5, 2, dz=1, n_combo=4, seed=46)
    h = make_hyper(p, seed=47)
    want = {-1: E.FP64_DMMA, E.FP64_INT8: E.FP64_INT8}   # by size, T = 9 < 24: DMMA
    E.pool_clear()
    prev = E.set_fp64_mode(-1)
    try:
        for order in ((-1, E.FP64_INT8), (E.FP64_INT8, -1)):
            nll = []
            for mode in order:
                E.set_fp64_mode(mode)
                eng = E.Engine(**engine_kwargs(p))   # the second create finds the first handle parked
                try:
                    assert eng.fp64_mode() == want[mode], (order, mode)
                    nll.append(eng.mll_grad(h, want_grad=True)["nll"])
                finally:
                    eng.close()
            assert abs(nll[0] - nll[1]) <= 1e-11 * abs(nll[1]), nll
        E.set_fp64_mode(-1)

        def launches_per_evaluation(chol, fresh):
            if fresh:
                E.pool_clear()
            if chol is None:
                monkeypatch.delenv("GPP_CHOL", raising=False)
            else:
                monkeypatch.setenv("GPP_CHOL", chol)
            eng = E.Engine(**engine_kwargs(p))
            try:
                eng.mll_grad(h, want_grad=True)
                before = E.launch_count()
                eng.mll_grad(h, want_grad=True)
                return E.launch_count() - before
            finally:
                eng.close()

        fresh = {c: launches_per_evaluation(c, True) for c in (None, "blocked")}
        assert fresh[None] != fresh["blocked"], fresh
        for order in ((None, "blocked"), ("blocked", None)):
            E.pool_clear()
            for c in order:
                assert launches_per_evaluation(c, False) == fresh[c], (order, c)
    finally:
        E.set_fp64_mode(prev)
        E.pool_clear()


def test_schedule_settings_stay_with_the_handle_created_under_them(monkeypatch):
    """A schedule switch belongs to the handle created under it: creating another handle with GPP_OVERLAP_INV=0
    changes neither the launches nor the likelihood of a handle that exists already, and once the variable is unset
    the next handle gets the default schedule again.  N = 2300 (T = 18) evaluates as a chain of launches (no graph
    replay), so the overlapped inverse changes the launches per evaluation."""
    from gpplus_b200 import _engine as E
    p = make_problem(2300, 5, 2, dz=2, n_combo=7, n_noise=2, seed=31)
    h = make_hyper(p, seed=13)

    def evaluate(eng):
        eng.mll_grad(h, want_grad=True)
        before = E.launch_count()
        nll = eng.mll_grad(h, want_grad=True)["nll"]
        return E.launch_count() - before, nll

    E.pool_clear()
    monkeypatch.delenv("GPP_OVERLAP_INV", raising=False)
    a = E.Engine(**engine_kwargs(p))
    try:
        count_a, nll_a = evaluate(a)
        monkeypatch.setenv("GPP_OVERLAP_INV", "0")
        b = E.Engine(**engine_kwargs(p))
        try:
            count_b = evaluate(b)[0]
        finally:
            b.close()   # parked under GPP_OVERLAP_INV=0
        assert count_b != count_a, count_a
        assert evaluate(a) == (count_a, nll_a)
        monkeypatch.delenv("GPP_OVERLAP_INV")
        c = E.Engine(**engine_kwargs(p))
        try:
            assert evaluate(c)[0] == count_a
        finally:
            c.close()
    finally:
        a.close()
        E.pool_clear()


@pytest.mark.parametrize("kernel,n,n_pass", [(0, 300, 3), (2, 517, 5), (1, 130, 2)])
def test_multi_pass_ensemble_covariance_matches_oracle(kernel, n, n_pass):
    """Multi-pass ensemble covariance of the probabilistic embedding (gp_plus.py:387-399, 474-482):
    K = (1/k) sum_p K(Z_p) over k latent tables -- dense K, NLL, every gradient (one block of d_z per table) and
    predictions against the CPU oracle."""
    from gpplus_b200 import _engine as E
    from oracle import gp_oracle as O
    p = make_problem(n=n, dq=4, kernel=kernel, dz=2, n_combo=7, n_noise=2, n_mean=2, seed=60 + n_pass, n_pass=n_pass)
    h = make_hyper(p, seed=70 + n_pass)
    eng = E.Engine(**engine_kwargs(p))
    try:
        ref = O.mll(p, h, want_grad=True, return_mats=True)
        K = eng.covariance(h)
        assert np.max(np.abs(K - ref["K"])) <= 1e-13
        out = eng.mll_grad(h, want_grad=True)
        assert abs(out["nll"] - ref["nll"]) <= 1e-9 * abs(ref["nll"])
        assert out["d_z"].shape == (n_pass, 7, 2)
        for k in ("d_w", "d_z", "d_noise", "d_beta"):
            err = np.max(np.abs(out[k] - ref[k])) / max(1e-300, np.max(np.abs(ref[k])))
            assert err < 1e-8, (k, err)
        assert abs(out["d_sigma_f2"] - ref["d_sigma_f2"]) <= 1e-8 * abs(ref["d_sigma_f2"])
        cand = make_candidates(p, 200, seed=80)
        eng.factorize(h)
        mu, var = eng.predict(cand["xq"], level_idx=cand["level_idx"], noise_idx=cand["noise_idx"],
                              mean_idx=cand["mean_idx"], include_noise=True)
        mu_r, var_r = O.predict(p, h, cand, include_noise=True)
        assert np.max(np.abs(mu - mu_r)) <= 1e-9 and np.max(np.abs(var - var_r)) <= 1e-9
    finally:
        eng.close()
