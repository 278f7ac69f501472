"""CPU reference for gpp_acq_qbatch: the t-batch posteriors of ``qbatch_posterior_reference``, the Monte-Carlo
utility (qEI, qNEI, qUCB) in torch with autograd through the per-block Cholesky factor, and the chain into that
reference's d_xq through (g_mean, g_cov)."""
import math
from typing import Dict, Optional

import numpy as np
import torch

from qbatch_posterior_reference import posterior_qbatch

KINDS = {"EI": 0, "NEI": 1, "UCB": 2}


def ladder_jitter(cov: torch.Tensor) -> torch.Tensor:
    """Per-block jitter of _compat._psd_safe_cholesky's ladder (0, 1e-8, 1e-7, 1e-6); NaN where every rung fails."""
    jit = torch.full(cov.shape[:-2], float("nan"), dtype=torch.float64)
    eye = torch.eye(cov.shape[-1], dtype=torch.float64)
    for j in (0.0, 1e-8, 1e-7, 1e-6):
        _, info = torch.linalg.cholesky_ex(cov + j * eye)
        jit = torch.where(torch.isnan(jit) & (info == 0), torch.full_like(jit, j), jit)
    return jit


def mc_utility(mean, cov, E, kind: int, best_f: float = 0.0, beta: float = 0.0, n_baseline: int = 0,
               maximize: bool = True, jitter: Optional[np.ndarray] = None):
    """(values [b], g_mean [b, q], g_cov [b, q, q], jitter [b]) of the utility averaged over the rows of E [S, q],
    shared by every t-batch; g_* are the gradients of sum(values) (torch's cholesky backward)."""
    mu = torch.as_tensor(np.asarray(mean), dtype=torch.float64).clone().requires_grad_(True)
    S = torch.as_tensor(np.asarray(cov), dtype=torch.float64).clone().requires_grad_(True)
    E = torch.as_tensor(np.asarray(E), dtype=torch.float64)
    q = mu.shape[-1]
    jit = ladder_jitter(S.detach()) if jitter is None else torch.as_tensor(np.asarray(jitter), dtype=torch.float64)
    sgn = 1.0 if maximize else -1.0
    with torch.enable_grad():
        L = torch.linalg.cholesky(S + jit[:, None, None] * torch.eye(q, dtype=torch.float64))
        y = mu[None] + torch.einsum("tij,sj->sti", L, E)  # [S, b, q]
        z = sgn * y
        if kind == KINDS["EI"]:
            u = (z.max(-1).values - sgn * best_f).clamp_min(0)
        elif kind == KINDS["NEI"]:
            qc = q - n_baseline
            u = (z[..., :qc].max(-1).values - z[..., qc:].max(-1).values).clamp_min(0)
        else:
            u = (sgn * mu[None] + math.sqrt(beta * math.pi / 2) * (y - mu[None]).abs()).max(-1).values
        v = u.mean(0)
        gm, gc = torch.autograd.grad(v.sum(), (mu, S))
    return v.detach().numpy(), gm.numpy(), gc.numpy(), jit.numpy()


def acq_qbatch(problem: Dict, hyper: Dict, cand: Dict, q_tot: int, kind: int, E, best_f: float = 0.0,
               beta: float = 0.0, n_baseline: int = 0, maximize: bool = True, include_noise: bool = False,
               jitter: Optional[np.ndarray] = None):
    """(values [b], d_xq [b*q_tot, dq], jitter [b]) in scaled y units for the t-batches of ``cand``."""
    mean, cov, _ = posterior_qbatch(problem, hyper, cand, q_tot, include_noise)
    v, gm, gc, jit = mc_utility(mean, cov, E, kind, best_f, beta, n_baseline, maximize, jitter)
    _, _, d = posterior_qbatch(problem, hyper, cand, q_tot, include_noise, gm, gc)
    return v, d, jit
