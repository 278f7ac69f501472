"""CPU reference for gpp_predict_grad, shared by the prediction-gradient tests: torch autograd through the dense
exact prediction of ``oracle.gp_oracle`` (covariance, psd_safe_cholesky, mean gather) w.r.t. the candidates'
quantitative inputs -- what GP_Plus.predict_with_grad hands back to Xtest (models/gp_plus.py:626-628)."""
from typing import Dict

import numpy as np
import torch

from oracle import gp_oracle as O


def predict_grad(problem: Dict, hyper: Dict, cand: Dict, include_noise: bool = False, min_var: float = 1e-10,
                 mode: str = "expansion"):
    """(mu, var, d_mu [m, dq], d_var [m, dq]) in SCALED y units; mu / var as ``oracle.gp_oracle.predict``.  Each
    candidate's outputs depend on its own row only, so the gradient of the sum is the per-candidate gradient; below
    min_var the variance is clamped and has no gradient (torch clamp_min)."""
    n, dq, xq, y, lvl, nidx, midx = O._problem_tensors(problem)
    kind = int(problem["kernel"])
    n_mean = int(problem.get("n_mean", 0))
    w, z, sf2, noise, beta = O._hyper_tensors(problem, hyper, False)
    m_c = int(cand["m"])
    xc = O._t(cand["xq"]).reshape(m_c, dq).clone().requires_grad_(True)
    lc = None if cand.get("level_idx") is None else torch.as_tensor(np.asarray(cand["level_idx"]), dtype=torch.long)
    centre = xq.mean(0, keepdim=True)
    with torch.no_grad():
        K = O.covariance(xq, lvl, xq, lvl, w, z, sf2, kind, mode, centre)
        L, _ = O.psd_safe_cholesky(K + torch.diag(noise[nidx]))
        alpha = torch.cholesky_solve((y - O._mean_vector(midx, beta, n_mean)).unsqueeze(-1), L)
    with torch.enable_grad():  # also when called where gradients are off (inside an autograd Function's forward)
        Ks = O.covariance(xc, lc, xq, lvl, w, z, sf2, kind, mode, centre)  # [m, n]
        cm = torch.zeros(m_c, dtype=torch.long) if cand.get("mean_idx") is None else torch.as_tensor(
            np.asarray(cand["mean_idx"]), dtype=torch.long)
        mu = O._mean_vector(cm, beta, n_mean) + (Ks @ alpha).squeeze(-1)
        V = torch.linalg.solve_triangular(L, Ks.T, upper=False)
        var = sf2 - (V * V).sum(0)
        if include_noise:
            cn = torch.zeros(m_c, dtype=torch.long) if cand.get("noise_idx") is None else torch.as_tensor(
                np.asarray(cand["noise_idx"]), dtype=torch.long)
            var = var + noise[cn]
        var = var.clamp_min(min_var)
        d_mu, d_var = torch.zeros_like(xc), torch.zeros_like(xc)
        if dq > 0:  # without quantitative inputs nothing depends on xc
            d_mu, = torch.autograd.grad(mu.sum(), xc, retain_graph=True)
            if var.requires_grad:
                d_var, = torch.autograd.grad(var.sum(), xc)
    return mu.detach().numpy(), var.detach().numpy(), d_mu.detach().numpy(), d_var.detach().numpy()
