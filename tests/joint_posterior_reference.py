"""CPU reference for gpp_predict_joint / gpp_sample_posterior, shared by the joint-posterior tests: the dense exact
joint predictive distribution assembled from ``oracle.gp_oracle`` (covariance, psd_safe_cholesky, mean gather), the
joint structure of the reference's ``GPR.posterior`` (gpregression.py:151-166)."""
from typing import Dict

import numpy as np
import torch

from oracle import gp_oracle as O


def predict_joint(problem: Dict, hyper: Dict, cand: Dict, include_noise: bool = False, mode: str = "expansion"):
    """(mu [m], Sigma* [m, m]) in SCALED y units: mu as ``oracle.gp_oracle.predict``,
    Sigma* = K** - K* K_y^-1 K*^T (+ diag(noise of each candidate's group)), not clamped."""
    n, dq, xq, y, lvl, nidx, midx = O._problem_tensors(problem)
    kind = int(problem["kernel"])
    n_mean = int(problem.get("n_mean", 0))
    with torch.no_grad():
        w, z, sf2, noise, beta = O._hyper_tensors(problem, hyper, False)
        m_c = int(cand["m"])
        xc = O._t(cand["xq"]).reshape(m_c, dq)
        lc = None if cand.get("level_idx") is None else torch.as_tensor(np.asarray(cand["level_idx"]), dtype=torch.long)
        centre = xq.mean(0, keepdim=True)
        K = O.covariance(xq, lvl, xq, lvl, w, z, sf2, kind, mode, centre)
        L, _ = O.psd_safe_cholesky(K + torch.diag(noise[nidx]))
        alpha = torch.cholesky_solve((y - O._mean_vector(midx, beta, n_mean)).unsqueeze(-1), L)
        Ks = O.covariance(xc, lc, xq, lvl, w, z, sf2, kind, mode, centre)  # [m, n]
        Kss = O.covariance(xc, lc, xc, lc, w, z, sf2, kind, mode, centre)  # [m, m]
        cm = torch.zeros(m_c, dtype=torch.long) if cand.get("mean_idx") is None else torch.as_tensor(
            np.asarray(cand["mean_idx"]), dtype=torch.long)
        mu = O._mean_vector(cm, beta, n_mean) + (Ks @ alpha).squeeze(-1)
        V = torch.linalg.solve_triangular(L, Ks.T, upper=False)  # [n, m]
        cov = Kss - V.T @ V
        # the diagonal of K** is sigma_f^2 exactly (distance 0), as in oracle.gp_oracle.predict's variance
        cov.diagonal().copy_(sf2 - (V * V).sum(0))
        if include_noise:
            cn = torch.zeros(m_c, dtype=torch.long) if cand.get("noise_idx") is None else torch.as_tensor(
                np.asarray(cand["noise_idx"]), dtype=torch.long)
            cov = cov + torch.diag(noise[cn])
        cov = 0.5 * (cov + cov.T)
    return mu.numpy(), cov.numpy()


def joint_factor(cov: np.ndarray):
    """(L*, jitter) of the joint covariance by the psd_safe_cholesky ladder."""
    L, jit = O.psd_safe_cholesky(torch.as_tensor(cov, dtype=torch.float64))
    return L.numpy(), jit
