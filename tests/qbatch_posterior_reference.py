"""CPU reference for gpp_posterior_qbatch / gpp_posterior_qbatch_grad, shared by the t-batch posterior tests: per
t-batch of q consecutive candidates, the dense exact joint posterior of ``joint_posterior_reference`` (covariance,
psd_safe_cholesky and mean gather of ``oracle.gp_oracle``), and torch autograd through it w.r.t. the candidates'
quantitative inputs as in ``predict_grad_reference``."""
from typing import Dict, Optional

import numpy as np
import torch

from oracle import gp_oracle as O


def posterior_qbatch(problem: Dict, hyper: Dict, cand: Dict, q: int, include_noise: bool = False,
                     g_mean: Optional[np.ndarray] = None, g_cov: Optional[np.ndarray] = None,
                     mode: str = "expansion", group: int = 256):
    """(mean [b, q], cov [b, q, q], d_xq [b*q, dq]) in SCALED y units for the b = m / q t-batches of ``cand``.
    Each block is K**_t - K*_t K_y^-1 K*_t^T with the diagonal sf2 - |L^-1 k*_i|^2 (+ noise of the row's group), made
    exactly symmetric, not clamped; d_xq = d/d xq of sum(g_mean * mean) + sum(g_cov * cov) (zero when neither is
    given).  t-batches are independent, so they are evaluated ``group`` at a time."""
    n, dq, xq, y, lvl, nidx, midx = O._problem_tensors(problem)
    kind = int(problem["kernel"])
    n_mean = int(problem.get("n_mean", 0))
    w, z, sf2, noise, beta = O._hyper_tensors(problem, hyper, False)
    m_c = int(cand["m"])
    b = m_c // q
    xc = O._t(cand["xq"]).reshape(m_c, dq)
    lc = None if cand.get("level_idx") is None else torch.as_tensor(np.asarray(cand["level_idx"]), dtype=torch.long)
    cm = torch.zeros(m_c, dtype=torch.long) if cand.get("mean_idx") is None else torch.as_tensor(
        np.asarray(cand["mean_idx"]), dtype=torch.long)
    cn = torch.zeros(m_c, dtype=torch.long) if cand.get("noise_idx") is None else torch.as_tensor(
        np.asarray(cand["noise_idx"]), dtype=torch.long)
    gm = None if g_mean is None else torch.as_tensor(np.asarray(g_mean), dtype=torch.float64).reshape(b, q)
    gc = None if g_cov is None else torch.as_tensor(np.asarray(g_cov), dtype=torch.float64).reshape(b, q, q)
    centre = xq.mean(0, keepdim=True)
    with torch.no_grad():
        K = O.covariance(xq, lvl, xq, lvl, w, z, sf2, kind, mode, centre)
        L, _ = O.psd_safe_cholesky(K + torch.diag(noise[nidx]))
        alpha = torch.cholesky_solve((y - O._mean_vector(midx, beta, n_mean)).unsqueeze(-1), L)
    eye = torch.eye(q, dtype=torch.float64)
    means, covs, grads = [], [], []
    for t0 in range(0, b, group):
        t1 = min(b, t0 + group)
        nb, r0, r1 = t1 - t0, t0 * q, t1 * q
        xg = xc[r0:r1].clone().requires_grad_(True)
        lg = None if lc is None else lc[r0:r1]
        with torch.enable_grad():
            Ks = O.covariance(xg, lg, xq, lvl, w, z, sf2, kind, mode, centre)  # [R, n]
            mu = O._mean_vector(cm[r0:r1], beta, n_mean) + (Ks @ alpha).squeeze(-1)
            V = torch.linalg.solve_triangular(L, Ks.T, upper=False).T.reshape(nb, q, n)
            Kss = O.covariance(xg, lg, xg, lg, w, z, sf2, kind, mode, centre)  # [R, R]
            idx = torch.arange(r1 - r0).reshape(nb, q)
            cov = Kss[idx[:, :, None], idx[:, None, :]] - V @ V.transpose(1, 2)
            diag = sf2 - (V * V).sum(-1)
            if include_noise:
                diag = diag + noise[cn[r0:r1]].reshape(nb, q)
            cov = cov * (1.0 - eye) + torch.diag_embed(diag)
            cov = 0.5 * (cov + cov.transpose(1, 2))
            mu = mu.reshape(nb, q)
            d = torch.zeros_like(xg)
            loss = None
            if gm is not None:
                loss = (gm[t0:t1] * mu).sum()
            if gc is not None:
                loss = (gc[t0:t1] * cov).sum() + (0.0 if loss is None else loss)
            if dq > 0 and loss is not None and loss.requires_grad:
                d, = torch.autograd.grad(loss, xg)
        means.append(mu.detach())
        covs.append(cov.detach())
        grads.append(d.detach())
    if b == 0:
        return np.zeros((0, q)), np.zeros((0, q, q)), np.zeros((0, dq))
    return torch.cat(means).numpy(), torch.cat(covs).numpy(), torch.cat(grads).numpy()
