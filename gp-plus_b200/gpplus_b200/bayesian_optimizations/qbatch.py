"""Proposing a batch of q points by maximising a batch acquisition (Monte-Carlo qEI, qNEI, qUCB, qNIPV, the one-shot
knowledge gradient, or GIBBON) of a fitted model: Sobol screening of raw t-batches, then one joint L-BFGS-B run over
the best restarts with the engine's gradients (GPR.acquisition_qbatch / gpp_acq_qbatch, gpp_nipv_qbatch;
GPR.knowledge_gradient / gpp_kg_qbatch; GPR.gibbon / gpp_gibbon_qbatch), and the maximiser of the posterior mean that
cost-aware knowledge gradient is measured against (GPR.predict / gpp_predict_grad)."""
from typing import Dict, Optional, Tuple

import numpy as np
import torch
from scipy.optimize import minimize

from ..models.gpregression import GPR, sobol_normal_samples


def _columns(model, bounds, fixed_columns, caller: str):
    """(d, quantitative columns, lower and upper bounds [dq], {column: value}) of an optimiser's arguments."""
    d = int(model.train_inputs[0].shape[1])
    cols = list(model._quant_columns())
    other = [c for c in range(d) if c not in cols]
    fixed = dict(fixed_columns or {})
    missing = [c for c in other if c not in fixed]
    if missing:
        raise ValueError("%s: columns %s are not quantitative and need fixed_columns" % (caller, missing))
    bad = [c for c in fixed if c in cols]
    if bad:
        raise ValueError("%s: columns %s are quantitative and cannot be fixed" % (caller, bad))
    lo, hi = (torch.as_tensor(np.asarray(bounds, dtype=np.float64)).reshape(2, -1)[k] for k in (0, 1))
    if lo.numel() != len(cols):
        raise ValueError("%s: bounds cover %d columns, the model has %d quantitative" % (caller, lo.numel(), len(cols)))
    if len(cols) == 0:
        raise ValueError("%s: the model has no quantitative column to optimise" % caller)
    return d, cols, lo, hi, fixed


def _multistart(value, full, cols, lo, hi, rows: int, num_restarts: int, raw_samples: int, options: Optional[dict],
                seed: int):
    """Sobol screening, then one joint L-BFGS-B run, of ``value`` (model inputs [k, rows, d] -> values [k]).

    ``raw_samples`` Sobol t-batches of quantitative inputs [rows, dq] inside [lo, hi] are scored in one values-only
    call; the best ``num_restarts`` (ties broken by index) are optimised jointly on minus the sum of their values.
    ``full`` maps quantitative inputs [k, rows, dq] to model inputs, whose quantitative columns are ``cols``.  Returns
    the best optimised t-batch [rows, d] and its value, and the best screened t-batch and its value."""
    dq = len(cols)
    raw = torch.quasirandom.SobolEngine(dimension=rows * dq, scramble=True, seed=int(seed)).draw(int(raw_samples),
                                                                                             dtype=torch.float64)
    z_raw = lo + (hi - lo) * raw.reshape(-1, rows, dq)
    with torch.no_grad():
        v_raw = value(full(z_raw)).double().numpy()
    k = min(int(num_restarts), z_raw.shape[0])
    order = np.lexsort((np.arange(len(v_raw)), -v_raw))[:k]  # best first, ties by index
    z0 = z_raw[torch.as_tensor(order)].numpy()

    def neg(flat):
        z = torch.tensor(flat.reshape(k, rows, dq), dtype=torch.float64)
        X = full(z).requires_grad_(True)
        v = value(X).sum()
        g, = torch.autograd.grad(v, X)
        return -float(v.detach()), -g[:, :, cols].numpy().reshape(-1).astype(np.float64)

    box = list(zip(np.tile(lo.numpy(), k * rows), np.tile(hi.numpy(), k * rows)))
    res = minimize(neg, z0.reshape(-1), jac=True, method="L-BFGS-B", bounds=box, options=options)
    z_opt = torch.tensor(np.clip(res.x.reshape(k, rows, dq), lo.numpy(), hi.numpy()), dtype=torch.float64)
    with torch.no_grad():
        v_opt = value(full(z_opt)).double().numpy()
    best = int(np.lexsort((np.arange(k), -v_opt))[0])
    return full(z_opt[best:best + 1])[0], float(v_opt[best]), full(z_raw[order[:1]])[0], float(v_raw[order[0]])


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
    d, cols, lo, hi, fixed = _columns(model, bounds, fixed_columns, "optimize_acquisition_qbatch")

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

    X, v, _, _ = _multistart(lambda X: model.acquisition_qbatch(X, kind, **acq_kwargs), full, cols, lo, hi, q,
                             num_restarts, raw_samples, options, seed)
    return X, v


def optimize_knowledge_gradient(model, bounds, q: int, num_fantasies: int = 64,
                                fixed_columns: Optional[Dict[int, float]] = None,
                                fantasy_fixed_columns: Optional[Dict[int, float]] = None, num_restarts: int = 8,
                                raw_samples: int = 256, options: Optional[dict] = None, seed: int = 0,
                                **kg_kwargs) -> Tuple[torch.Tensor, float]:
    """Best batch ``X`` [q, d] of the one-shot knowledge gradient ``model.knowledge_gradient`` and its value.

    The q actual rows and the ``num_fantasies`` fantasy solutions are optimised jointly, as botorch's one-shot qKG
    does, and only the actual rows are returned.  ``bounds``, ``fixed_columns``, the screening and the L-BFGS-B run are
    those of ``optimize_acquisition_qbatch``.  ``fantasy_fixed_columns`` overrides ``fixed_columns`` on the fantasy
    rows: ``{source_column: target_source}`` projects the fantasy solutions to the target fidelity, as botorch's
    qMultiFidelityKnowledgeGradient does.  The base samples are drawn once from ``seed`` unless ``base_samples`` is
    given; ``kg_kwargs`` (``maximize``, ``current_value``, ``cost_by_source``) go to ``knowledge_gradient``.  The
    value returned is that of the best optimised batch, or of the best screened one when that is higher."""
    q, nf = int(q), int(num_fantasies)
    rows = q + nf
    d, cols, lo, hi, fixed = _columns(model, bounds, fixed_columns, "optimize_knowledge_gradient")
    ffixed = dict(fixed)
    ffixed.update(fantasy_fixed_columns or {})
    bad = [c for c in ffixed if c in cols]
    if bad:
        raise ValueError("optimize_knowledge_gradient: columns %s are quantitative and cannot be fixed" % bad)
    kg_kwargs = dict(kg_kwargs)
    if kg_kwargs.get("base_samples") is None:
        kg_kwargs["base_samples"] = sobol_normal_samples(nf, q, seed)

    def full(z: torch.Tensor) -> torch.Tensor:  # quantitative inputs [k, q + F, dq] -> model inputs [k, q + F, d]
        X = torch.zeros(z.shape[0], rows, d, dtype=torch.float64)
        X[:, :, cols] = z
        for c, v in fixed.items():
            X[:, :q, c] = float(v)
        for c, v in ffixed.items():
            X[:, q:, c] = float(v)
        return X

    X, v, X_raw, v_raw = _multistart(lambda X: model.knowledge_gradient(X, nf, **kg_kwargs), full, cols, lo, hi,
                                     rows, num_restarts, raw_samples, options, seed)
    if v_raw > v:
        X, v = X_raw, v_raw
    return X[:q], v


def optimize_posterior_mean(model, bounds, fixed_columns: Optional[Dict[int, float]] = None, maximize: bool = True,
                            num_restarts: int = 8, raw_samples: int = 256, options: Optional[dict] = None,
                            seed: int = 0) -> Tuple[torch.Tensor, float]:
    """Point ``x`` [d] that maximises sigma times the posterior mean (sigma = +1 to maximise, -1 to minimise) in the
    original y units, and that value: botorch's PosteriorMean under FixedFeatureAcquisitionFunction.  With
    ``fixed_columns`` holding the source column at the target fidelity it gives the ``current_value`` of cost-aware
    knowledge gradient.  Screening and L-BFGS-B as ``optimize_acquisition_qbatch``, on GPR.predict with input
    gradients (gpp_predict_grad)."""
    d, cols, lo, hi, fixed = _columns(model, bounds, fixed_columns, "optimize_posterior_mean")
    sgn = 1.0 if maximize else -1.0

    def full(z: torch.Tensor) -> torch.Tensor:  # quantitative inputs [k, 1, dq] -> model inputs [k, 1, d]
        X = torch.zeros(z.shape[0], 1, d, dtype=torch.float64)
        X[:, :, cols] = z
        for c, v in fixed.items():
            X[:, :, c] = float(v)
        return X

    def value(X: torch.Tensor) -> torch.Tensor:
        return sgn * GPR.predict(model, X[:, 0, :]).double()

    X, v, X_raw, v_raw = _multistart(value, full, cols, lo, hi, 1, num_restarts, raw_samples, options, seed)
    if v_raw > v:
        X, v = X_raw, v_raw
    return X[0], v


def optimize_gibbon(model, bounds, q: int, max_values, fixed_columns: Optional[Dict[int, float]] = None,
                    target_fixed_columns: Optional[Dict[int, float]] = None, cost_by_source=None, sources=None,
                    sequential: bool = True, num_restarts: int = 8, raw_samples: int = 256,
                    options: Optional[dict] = None, seed: int = 0, maximize: bool = True) -> Tuple[torch.Tensor, float]:
    """Batch ``X`` [q, d] chosen by GIBBON (``model.gibbon`` with ``max_values``, ``maximize``,
    ``target_fixed_columns`` and ``cost_by_source``), and ``model.gibbon`` of that batch (per unit cost when costs are
    given).

    ``sequential=True`` is botorch's recommended greedy mode: q steps, each a one-row screening and L-BFGS-B run (as
    ``optimize_acquisition_qbatch``, seed ``seed + step``) on the gain over the earlier picks, passed as ``X_pending``.
    ``sources`` (sequential only) runs one such search per listed value of the source column (the last column) at
    every step and keeps the pick with the highest gain per unit cost; ties go to the first listed source.
    ``sequential=False`` optimises the q rows jointly in one run.  ``bounds`` and ``fixed_columns`` are those of
    ``optimize_acquisition_qbatch``; a search's best screened row replaces its optimised one when it scores higher."""
    q = int(q)
    if q < 1:
        raise ValueError("optimize_gibbon: q must be >= 1, got %d" % q)
    fixed_columns = dict(fixed_columns or {})
    if sources is not None:
        if not sequential:
            raise ValueError("optimize_gibbon: sources needs sequential=True")
        if len(sources) == 0:
            raise ValueError("optimize_gibbon: sources is empty")
        last = int(model.train_inputs[0].shape[1]) - 1
        if last in model._quant_columns():
            raise ValueError("optimize_gibbon: sources needs a source column (the last), not a quantitative one")
        fixed_columns.setdefault(last, float(sources[0]))  # the source column is set per search
    d, cols, lo, hi, fixed = _columns(model, bounds, fixed_columns, "optimize_gibbon")
    kw = dict(maximize=maximize, target_fixed_columns=target_fixed_columns, cost_by_source=cost_by_source)

    def full_with(fx: Dict[int, float], rows: int):
        def full(z: torch.Tensor) -> torch.Tensor:  # quantitative inputs [k, rows, dq] -> model inputs [k, rows, d]
            X = torch.zeros(z.shape[0], rows, d, dtype=torch.float64)
            X[:, :, cols] = z
            for c, v in fx.items():
                X[:, :, c] = float(v)
            return X
        return full

    def search(fx: Dict[int, float], rows: int, pending: Optional[torch.Tensor], step_seed: int):
        X, v, X_raw, v_raw = _multistart(lambda X: model.gibbon(X, max_values, X_pending=pending, **kw),
                                         full_with(fx, rows), cols, lo, hi, rows, num_restarts, raw_samples, options,
                                         step_seed)
        return (X_raw, v_raw) if v_raw > v else (X, v)

    if sequential:
        picks = []
        for step in range(q):
            pending = torch.stack(picks) if picks else None
            best = None
            for src in (sources if sources is not None else [None]):
                fx = dict(fixed)
                if src is not None:
                    fx[d - 1] = float(src)
                X1, v1 = search(fx, 1, pending, int(seed) + step)
                if best is None or v1 > best[1]:
                    best = (X1[0], v1)
            picks.append(best[0])
        X = torch.stack(picks)
    else:
        X, _ = search(fixed, q, None, int(seed))
    with torch.no_grad():
        v = float(model.gibbon(X[None], max_values, **kw)[0])
    return X, v
