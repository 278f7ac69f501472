"""CPU reference for gpp_kg_qbatch: the one-shot knowledge gradient in closed form on the t-batch posteriors of
``qbatch_posterior_reference`` (with every row's noise), in torch with autograd through the per-block Cholesky factor
and chained into that reference's d_xq through (g_mean, g_cov); plus the literal semantics of botorch's one-shot qKG
with the PosteriorMean value function (append the actual points with fantasised observations to the training set,
refactorise, take the posterior mean at the fantasy solution) that the closed form must equal."""
from typing import Dict, Optional

import numpy as np
import torch

from oracle import gp_oracle as O
from qacq_reference import ladder_jitter
from qbatch_posterior_reference import posterior_qbatch


def kg_block(mean, cov, q: int, E, maximize: bool = True, jitter: Optional[np.ndarray] = None):
    """(values [b], g_mean [b, q_tot], g_cov [b, q_tot, q_tot], jitter [b]) of the closed form on blocks of
    q_tot = q + F rows (actual rows first); E [F, q]; g_* are the gradients of sum(values)."""
    mu = torch.as_tensor(np.asarray(mean), dtype=torch.float64).clone().requires_grad_(True)
    S = torch.as_tensor(np.asarray(cov), dtype=torch.float64).clone().requires_grad_(True)
    E = torch.as_tensor(np.asarray(E), dtype=torch.float64)
    sgn = 1.0 if maximize else -1.0
    A0 = S.detach()[:, :q, :q]
    jit = ladder_jitter(A0) if jitter is None else torch.as_tensor(np.asarray(jitter), dtype=torch.float64)
    with torch.enable_grad():
        L = torch.linalg.cholesky(S[:, :q, :q] + jit[:, None, None] * torch.eye(q, dtype=torch.float64))
        W = torch.linalg.solve_triangular(L, S[:, :q, q:], upper=False)  # [b, q, F]: w_f = L^-1 c_f
        v = (sgn * (mu[:, q:] + torch.einsum("tif,fi->tf", W, E))).mean(-1)
        gm, gc = torch.autograd.grad(v.sum(), (mu, S))
    return v.detach().numpy(), gm.numpy(), gc.numpy(), jit.numpy()


def kg_qbatch(problem: Dict, hyper: Dict, cand: Dict, q: int, n_fantasies: int, E, maximize: bool = True,
              jitter: Optional[np.ndarray] = None):
    """(values [b], d_xq [b*q_tot, dq], jitter [b]) in scaled y units for the t-batches of q + n_fantasies rows of
    ``cand``."""
    q_tot = q + n_fantasies
    mean, cov, _ = posterior_qbatch(problem, hyper, cand, q_tot, True)
    v, gm, gc, jit = kg_block(mean, cov, q, E, maximize, jitter)
    _, _, d = posterior_qbatch(problem, hyper, cand, q_tot, True, gm, gc)
    return v, d, jit


def kg_refit(problem: Dict, hyper: Dict, cand: Dict, q: int, n_fantasies: int, E, maximize: bool = True,
             jitter: Optional[np.ndarray] = None, mode: str = "expansion") -> np.ndarray:
    """values [b] by botorch's semantics: for every t-batch and fantasy f, the exact GP on the training set and the q
    actual points, observed at y_f = mu + L e_f each with its group's noise, refactorised densely, and its posterior
    mean at fantasy solution f; sigma times their mean over f.  The ladder's jitter j_t, which the closed form adds to
    A_t, is added to the actual points' noise here, the same model."""
    n, dq, xq, y, lvl, nidx, midx = O._problem_tensors(problem)
    kind = int(problem["kernel"])
    n_mean = int(problem.get("n_mean", 0))
    w, z, sf2, noise, beta = O._hyper_tensors(problem, hyper, False)
    centre = xq.mean(0, keepdim=True)
    q_tot = q + n_fantasies
    b = int(cand["m"]) // q_tot
    xc = O._t(cand["xq"]).reshape(-1, dq)
    lc = None if cand.get("level_idx") is None else torch.as_tensor(np.asarray(cand["level_idx"]), dtype=torch.long)
    cn = torch.zeros(b * q_tot, dtype=torch.long) if cand.get("noise_idx") is None else torch.as_tensor(
        np.asarray(cand["noise_idx"]), dtype=torch.long)
    cm = torch.zeros(b * q_tot, dtype=torch.long) if cand.get("mean_idx") is None else torch.as_tensor(
        np.asarray(cand["mean_idx"]), dtype=torch.long)
    E = torch.as_tensor(np.asarray(E), dtype=torch.float64)
    mean, cov, _ = posterior_qbatch(problem, hyper, cand, q_tot, True)
    mean, cov = torch.as_tensor(mean), torch.as_tensor(cov)
    jit = ladder_jitter(cov[:, :q, :q]) if jitter is None else torch.as_tensor(np.asarray(jitter), dtype=torch.float64)
    sgn = 1.0 if maximize else -1.0
    out = np.empty(b)
    for t in range(b):
        a = slice(t * q_tot, t * q_tot + q)
        fs = slice(t * q_tot + q, (t + 1) * q_tot)
        xa = torch.cat([xq, xc[a]])
        la = None if lvl is None else torch.cat([lvl, lc[a]])
        na = torch.cat([noise[nidx], noise[cn[a]] + jit[t]])
        ma = torch.cat([O._mean_vector(midx, beta, n_mean), O._mean_vector(cm[a], beta, n_mean)])
        L = torch.linalg.cholesky(O.covariance(xa, la, xa, la, w, z, sf2, kind, mode, centre) + torch.diag(na))
        Lt = torch.linalg.cholesky(cov[t, :q, :q] + jit[t] * torch.eye(q, dtype=torch.float64))
        Ks = O.covariance(xc[fs], None if lc is None else lc[fs], xa, la, w, z, sf2, kind, mode, centre)  # [F, n+q]
        mf = O._mean_vector(cm[fs], beta, n_mean)
        terms = []
        for f in range(n_fantasies):
            ya = torch.cat([y, mean[t, :q] + Lt @ E[f]])
            alpha = torch.cholesky_solve((ya - ma).unsqueeze(-1), L).squeeze(-1)
            terms.append(sgn * float(mf[f] + Ks[f] @ alpha))
        out[t] = float(np.mean(terms))
    return out
