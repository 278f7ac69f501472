"""CPU reference for gpp_gibbon_qbatch and gpp_max_value_quartiles: GIBBON in torch on the latent t-batch posteriors
of ``qbatch_posterior_reference``, with autograd through the per-block Cholesky factor chained into that reference's
d_xq through (g_mean, g_cov); and the max-value quartiles by bisection on torch.special.log_ndtr."""
import math
from typing import Dict, Optional

import numpy as np
import torch

from oracle import gp_oracle as O
from qacq_reference import ladder_jitter
from qbatch_posterior_reference import posterior_qbatch

EPS = 1e-8  # botorch's CLAMP_LB


def quality(v, s2, c, smu, mv, eps: float = EPS):
    """Q [...] of rows with observation variance v, target variance s2, cross-covariance c and sigma times the target
    mean smu (tensors of one shape), against max values mv [K]: -(1/2K) sum_k log max(1 - rho^2 r (gamma + r), eps)."""
    v, s2 = v.clamp_min(eps), s2.clamp_min(eps)
    rho2 = c * c / (v * s2)
    gamma = (mv - smu.unsqueeze(-1)) / s2.sqrt().unsqueeze(-1)
    # Phi as exp(log_ndtr): torch's Normal.cdf (0.5 (1 + erf)) and, on the CPU, torch.special.ndtr lose digits of
    # Phi(gamma) in the lower tail (1e-7 and 1e-10 relative at gamma = -6)
    r = torch.exp(-0.5 * gamma * gamma) / math.sqrt(2.0 * math.pi) / torch.special.log_ndtr(gamma).exp().clamp_min(eps)
    inner = (1.0 - rho2.unsqueeze(-1) * r * (gamma + r)).clamp_min(eps)
    return -0.5 * torch.log(inner).mean(-1)


def gibbon_block(mean, cov, noise, q: int, projected: bool, mv, maximize: bool = True,
                 jitter: Optional[np.ndarray] = None):
    """(values [b], g_mean [b, q_tot], g_cov [b, q_tot, q_tot], jitter [b]) of GIBBON on latent blocks of q_tot rows
    (the q actual rows first, then with ``projected`` their target copies); noise [b, q] of the actual rows; mv [K] in
    scaled units; g_* are the gradients of sum(values)."""
    mu = torch.as_tensor(np.asarray(mean), dtype=torch.float64).clone().requires_grad_(True)
    S = torch.as_tensor(np.asarray(cov), dtype=torch.float64).clone().requires_grad_(True)
    nz = torch.as_tensor(np.asarray(noise), dtype=torch.float64)
    mv = torch.as_tensor(np.asarray(mv), dtype=torch.float64).reshape(-1)
    sgn = 1.0 if maximize else -1.0
    tau = torch.arange(q) + (q if projected else 0)
    eye = torch.eye(q, dtype=torch.float64)
    V0 = S.detach()[:, :q, :q] + torch.diag_embed(nz)
    jit = ladder_jitter(V0) if jitter is None else torch.as_tensor(np.asarray(jitter), dtype=torch.float64)
    with torch.enable_grad():
        V = S[:, :q, :q] + torch.diag_embed(nz)
        A = V + jit[:, None, None] * eye
        L = torch.linalg.cholesky(A)
        D = (torch.log(torch.diagonal(L, dim1=-2, dim2=-1)) - 0.5 * torch.log(torch.diagonal(A, dim1=-2, dim2=-1))).sum(-1)
        v = torch.diagonal(V, dim1=-2, dim2=-1)
        s2 = S[:, tau, tau]
        c = S[:, torch.arange(q), tau]
        Q = quality(v, s2, c, sgn * mu[:, tau], mv).sum(-1)
        val = D + Q
        gm, gc = torch.autograd.grad(val.sum(), (mu, S))
    return val.detach().numpy(), gm.numpy(), gc.numpy(), jit.numpy()


def row_noise(hyper: Dict, cand: Dict, q_tot: int, q: int) -> np.ndarray:
    """[b, q] noise of the actual rows' groups (group 0 without noise_idx)."""
    m = int(cand["m"])
    nidx = np.zeros(m, dtype=np.int64) if cand.get("noise_idx") is None else np.asarray(cand["noise_idx"])
    return np.asarray(hyper["noise"], dtype=np.float64).reshape(-1)[nidx].reshape(-1, q_tot)[:, :q]


def gibbon_qbatch(problem: Dict, hyper: Dict, cand: Dict, q: int, projected: bool, mv, maximize: bool = True,
                  jitter: Optional[np.ndarray] = None):
    """(values [b], d_xq [b*q_tot, dq], jitter [b]) of the t-batches of q_tot = q (2q when ``projected``) rows of
    ``cand``; values in nats, mv in scaled units."""
    q_tot = 2 * q if projected else q
    mean, cov, _ = posterior_qbatch(problem, hyper, cand, q_tot, False)
    v, gm, gc, jit = gibbon_block(mean, cov, row_noise(hyper, cand, q_tot, q), q, projected, mv, maximize, jitter)
    _, _, d = posterior_qbatch(problem, hyper, cand, q_tot, False, gm, gc)
    return v, d, jit


def _loglik(y: float, smu: torch.Tensor, sd: torch.Tensor) -> float:
    return float(torch.special.log_ndtr((y - smu) / sd).sum())


def quartile_bracket(mean, var, maximize: bool = True):
    """(lo, hi) of gpp_max_value_quartiles: min sigma mu - 5 max s, max sigma mu + 5 max s, hi doubled away from lo
    while l(hi) < log 3/4; plus sigma mu and s."""
    smu = (1.0 if maximize else -1.0) * torch.as_tensor(np.asarray(mean), dtype=torch.float64)
    sd = torch.as_tensor(np.asarray(var), dtype=torch.float64).sqrt()
    lo = float(smu.min()) - 5.0 * float(sd.max())
    hi = float(smu.max()) + 5.0 * float(sd.max())
    while _loglik(hi, smu, sd) < math.log(0.75):
        hi = hi + (hi - lo)
    return lo, hi, smu, sd


def max_value_quartiles(mean, var, maximize: bool = True, steps: int = 40):
    """(quartiles [3], lo, hi): l(y) = sum_j log Phi((y - sigma mu_j) / s_j) = log p, p = 1/4, 1/2, 3/4, by ``steps``
    bisection steps of [lo, hi]; each quartile is the middle of its last bracket."""
    lo, hi, smu, sd = quartile_bracket(mean, var, maximize)
    out = []
    for p in (0.25, 0.5, 0.75):
        a, b = lo, hi
        for _ in range(steps):
            mid = 0.5 * (a + b)
            if _loglik(mid, smu, sd) < math.log(p):
                a = mid
            else:
                b = mid
        out.append(0.5 * (a + b))
    return np.array(out), lo, hi


def gumbel_from_quartiles(y1: float, y2: float, y3: float):
    """(alpha, beta) of the Gumbel fit of botorch's _sample_max_value_Gumbel."""
    beta = (y1 - y3) / (math.log(math.log(4.0 / 3.0)) - math.log(math.log(4.0)))
    return y2 + beta * math.log(math.log(2.0)), beta
