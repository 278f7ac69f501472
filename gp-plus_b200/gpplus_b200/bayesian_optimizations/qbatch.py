"""Proposing a batch of q points by maximising a batch acquisition (Monte-Carlo qEI, qNEI, qUCB, or qNIPV) of a
fitted model: Sobol screening of raw t-batches, then one joint L-BFGS-B run over the best restarts with the engine's
gradients (GPR.acquisition_qbatch / gpp_acq_qbatch, gpp_nipv_qbatch)."""
from typing import Dict, Optional, Tuple

import numpy as np
import torch
from scipy.optimize import minimize

from ..models.gpregression import sobol_normal_samples


def optimize_acquisition_qbatch(model, bounds, q: int, kind: str, fixed_columns: Optional[Dict[int, float]] = None,
                                num_restarts: int = 8, raw_samples: int = 256, options: Optional[dict] = None,
                                seed: int = 0, **acq_kwargs) -> Tuple[torch.Tensor, float]:
    """Best batch ``X`` [q, d] of ``model.acquisition_qbatch(X, kind, **acq_kwargs)`` and its value.

    ``bounds`` [2, dq] bounds the quantitative columns; the categorical and source columns are held at
    ``fixed_columns`` ({column: value}, required when the model has such columns).  ``raw_samples`` Sobol t-batches
    inside the bounds are scored in one values-only call; the best ``num_restarts`` (ties broken by index) are
    optimised jointly by one L-BFGS-B run on minus the sum of their values, with the same base samples throughout
    (drawn once from ``seed`` unless ``base_samples`` is given; qNIPV, which needs ``mc_points``, draws none).  ``options`` go to ``scipy.optimize.minimize``."""
    q = int(q)
    d = int(model.train_inputs[0].shape[1])
    cols = list(model._quant_columns())
    other = [c for c in range(d) if c not in cols]
    fixed = dict(fixed_columns or {})
    missing = [c for c in other if c not in fixed]
    if missing:
        raise ValueError("optimize_acquisition_qbatch: columns %s are not quantitative and need fixed_columns" % missing)
    bad = [c for c in fixed if c in cols]
    if bad:
        raise ValueError("optimize_acquisition_qbatch: columns %s are quantitative and cannot be fixed" % bad)
    lo, hi = (torch.as_tensor(np.asarray(bounds, dtype=np.float64)).reshape(2, -1)[k] for k in (0, 1))
    dq = len(cols)
    if lo.numel() != dq:
        raise ValueError("optimize_acquisition_qbatch: bounds cover %d columns, the model has %d quantitative"
                         % (lo.numel(), dq))
    if dq == 0:
        raise ValueError("optimize_acquisition_qbatch: the model has no quantitative column to optimise")

    acq_kwargs = dict(acq_kwargs)
    if kind != "qNIPV" and acq_kwargs.get("base_samples") is None:  # qNIPV is exact: no base samples
        n_b = 0
        if acq_kwargs.get("X_baseline") is not None:
            n_b = int(torch.as_tensor(acq_kwargs["X_baseline"]).reshape(-1, d).shape[0])
        acq_kwargs["base_samples"] = sobol_normal_samples(acq_kwargs.pop("num_samples", 512), q + n_b, seed)
    acq_kwargs.pop("num_samples", None)

    def full(z: torch.Tensor) -> torch.Tensor:  # quantitative inputs [k, q, dq] -> model inputs [k, q, d]
        X = torch.zeros(z.shape[0], q, d, dtype=torch.float64)
        X[:, :, cols] = z
        for c, v in fixed.items():
            X[:, :, c] = float(v)
        return X

    raw = torch.quasirandom.SobolEngine(dimension=q * dq, scramble=True, seed=int(seed)).draw(int(raw_samples),
                                                                                          dtype=torch.float64)
    z_raw = lo + (hi - lo) * raw.reshape(-1, q, dq)
    with torch.no_grad():
        v_raw = model.acquisition_qbatch(full(z_raw), kind, **acq_kwargs).double().numpy()
    k = min(int(num_restarts), z_raw.shape[0])
    order = np.lexsort((np.arange(len(v_raw)), -v_raw))[:k]  # best first, ties by index
    z0 = z_raw[torch.as_tensor(order)].numpy()

    def neg(flat):
        z = torch.tensor(flat.reshape(k, q, dq), dtype=torch.float64)
        X = full(z).requires_grad_(True)
        v = model.acquisition_qbatch(X, kind, **acq_kwargs).sum()
        g, = torch.autograd.grad(v, X)
        return -float(v.detach()), -g[:, :, cols].numpy().reshape(-1).astype(np.float64)

    box = list(zip(np.tile(lo.numpy(), k * q), np.tile(hi.numpy(), k * q)))
    res = minimize(neg, z0.reshape(-1), jac=True, method="L-BFGS-B", bounds=box, options=options)
    z_opt = torch.tensor(np.clip(res.x.reshape(k, q, dq), lo.numpy(), hi.numpy()), dtype=torch.float64)
    with torch.no_grad():
        v_opt = model.acquisition_qbatch(full(z_opt), kind, **acq_kwargs).double().numpy()
    best = int(np.lexsort((np.arange(k), -v_opt))[0])
    return full(z_opt[best:best + 1])[0], float(v_opt[best])
