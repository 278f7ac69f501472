"""CPU reference for gpp_ipv_points / gpp_nipv_qbatch: per t-batch, the dense joint posterior of [X_t; X_I] from
``qbatch_posterior_reference`` (no noise), the closed form of the negative integrated posterior variance in torch,
and the chain into that reference's d_xq through g_cov; plus the literal semantics of botorch's qNIPV (refactorise
the GP on the training set and the fantasy points, average the latent variance over X_I) that the closed form must
equal."""
from typing import Dict, Optional

import numpy as np
import torch

from oracle import gp_oracle as O
from qacq_reference import ladder_jitter
from qbatch_posterior_reference import posterior_qbatch


def _stacked(cand: Dict, ipv: Dict, q: int) -> Dict:
    """Candidates [b * (q + M)]: every t-batch's q rows followed by the M integration points."""
    b = int(cand["m"]) // q
    M = int(ipv["m"])
    xq = np.concatenate([np.concatenate([np.asarray(cand["xq"])[t * q:(t + 1) * q], np.asarray(ipv["xq"])])
                         for t in range(b)]) if b else np.zeros((0, np.asarray(cand["xq"]).shape[1]))
    lc, li = cand.get("level_idx"), ipv.get("level_idx")
    lvl = None
    if lc is not None:
        lvl = np.concatenate([np.concatenate([np.asarray(lc)[t * q:(t + 1) * q], np.asarray(li)]) for t in range(b)])
    return {"m": b * (q + M), "xq": xq, "level_idx": lvl, "noise_idx": None, "mean_idx": None}


def nipv_qbatch(problem: Dict, hyper: Dict, cand: Dict, ipv: Dict, q: int, jitter: Optional[np.ndarray] = None,
                group_rows: int = 2048):
    """(values [b], d_xq [b*q, dq], jitter [b]) in SCALED y units for the t-batches of ``cand`` against the integration
    points ``ipv`` ({"m", "xq", "level_idx"}).  Each t-batch is fantasised with the noise of its rows' groups
    (``cand["noise_idx"]``, group 0 when absent) and the psd_safe_cholesky ladder on A_t."""
    b = int(cand["m"]) // q
    M = int(ipv["m"])
    w, z, sf2, noise, beta = O._hyper_tensors(problem, hyper, False)
    cn = torch.zeros(b * q, dtype=torch.long) if cand.get("noise_idx") is None else torch.as_tensor(
        np.asarray(cand["noise_idx"]), dtype=torch.long)
    Q = q + M
    group = max(1, group_rows // Q)  # the reference forms K** over all rows of a group
    vals, grads, jits = [], [], []
    for t0 in range(0, b, group):
        t1 = min(b, t0 + group)
        sub = {k: (v[t0 * q:t1 * q] if isinstance(v, np.ndarray) else v) for k, v in cand.items()}
        sub["m"] = (t1 - t0) * q
        st = _stacked(sub, ipv, q)
        _, P, _ = posterior_qbatch(problem, hyper, st, Q, False)
        P = torch.as_tensor(P).clone().requires_grad_(True)
        nz = noise.detach()[cn[t0 * q:t1 * q]].reshape(t1 - t0, q)
        with torch.enable_grad():
            S = P[:, :q, :q] + torch.diag_embed(nz)
            jit = ladder_jitter(S.detach()) if jitter is None else torch.as_tensor(
                np.asarray(jitter)[t0:t1], dtype=torch.float64)
            A = S + jit[:, None, None] * torch.eye(q, dtype=torch.float64)
            C = P[:, q:, :q]  # [nb, M, q]
            vI = torch.diagonal(P[:, q:, q:], dim1=-2, dim2=-1)
            L = torch.linalg.cholesky(A)
            Z = torch.linalg.solve_triangular(L, C.transpose(1, 2), upper=False)  # L^-1 C^T
            v = -vI.mean(-1) + (Z * Z).sum((-2, -1)) / M
            gc, = torch.autograd.grad(v.sum(), P)
        _, _, d = posterior_qbatch(problem, hyper, st, Q, False, None, gc.numpy())
        vals.append(v.detach().numpy())
        jits.append(jit.numpy())
        grads.append(np.asarray(d).reshape(t1 - t0, Q, -1)[:, :q].reshape((t1 - t0) * q, -1))
    if b == 0:
        return np.zeros(0), np.zeros((0, int(problem["dq"]))), np.zeros(0)
    return np.concatenate(vals), np.concatenate(grads), np.concatenate(jits)


def nipv_refit(problem: Dict, hyper: Dict, cand: Dict, ipv: Dict, q: int, mode: str = "expansion") -> np.ndarray:
    """values [b] by botorch's semantics: the exact GP on the training set and X_t (any y, each row with its group's
    noise), refactorised per t-batch, and minus its latent variance averaged over the integration points."""
    n, dq, xq, _, lvl, nidx, _ = O._problem_tensors(problem)
    kind = int(problem["kernel"])
    w, z, sf2, noise, _ = O._hyper_tensors(problem, hyper, False)
    centre = xq.mean(0, keepdim=True)
    b = int(cand["m"]) // q
    xc = O._t(cand["xq"]).reshape(-1, dq)
    lc = None if cand.get("level_idx") is None else torch.as_tensor(np.asarray(cand["level_idx"]), dtype=torch.long)
    cn = torch.zeros(b * q, dtype=torch.long) if cand.get("noise_idx") is None else torch.as_tensor(
        np.asarray(cand["noise_idx"]), dtype=torch.long)
    xi = O._t(ipv["xq"]).reshape(-1, dq)
    li = None if ipv.get("level_idx") is None else torch.as_tensor(np.asarray(ipv["level_idx"]), dtype=torch.long)
    out = np.empty(b)
    for t in range(b):
        r = slice(t * q, (t + 1) * q)
        xa = torch.cat([xq, xc[r]])
        la = None if lvl is None else torch.cat([lvl, lc[r]])
        na = torch.cat([noise[nidx], noise[cn[r]]])
        K = O.covariance(xa, la, xa, la, w, z, sf2, kind, mode, centre) + torch.diag(na)
        L, _ = O.psd_safe_cholesky(K)
        Ks = O.covariance(xi, li, xa, la, w, z, sf2, kind, mode, centre)
        V = torch.linalg.solve_triangular(L, Ks.T, upper=False)
        out[t] = -float((sf2 - (V * V).sum(0)).mean())
    return out
