"""``GPR``: exact GP regression model backed by the B200 engine.

Mirrors models/gpregression.py:38-175 of the reference (constructor arguments, y min-max scaling,
noise constraint and priors, ``ScaleKernel`` wrapping, ``predict`` contract).  The reference builds
on gpytorch's ``ExactGP``; here the model only owns the raw hyper-parameters and the static training
data, and every O(N^2)/O(N^3) step -- covariance, Cholesky, alpha / log|K|, gradient, predictive
mean / variance -- is a call into ``libgpplus_b200.so``.
"""
from __future__ import annotations

import contextlib

import math
import threading
import warnings
from typing import List, Optional, Tuple, Union

import numpy as np
import torch
from torch.autograd.function import once_differentiable

from .. import _engine, kernels
from .._compat import (ConstantMean, GaussianLikelihood, GreaterThan, Kernel, LogNormalPrior, Module,
                       MultivariateNormal, NumericalWarning, Positive, ZeroMean, settings)
from ..likelihoods_noise.multifidelity import Multifidelity_likelihood
from ..priors import LogHalfHorseshoePrior, MollifiedUniformPrior
from ..utils.transforms import inv_softplus, softplus

_default_device = threading.local()


def set_default_device(index: int):
    """GPU index new engines of this thread are created on (restart workers pin one GPU each)."""
    _default_device.index = int(index)


def get_default_device() -> int:
    return getattr(_default_device, "index", 0)


class _EngineLogProb(torch.autograd.Function):
    """log N(y_scaled; m, K + noise) evaluated on the GPU; backward hands the fused analytic gradient
    (csrc/cov.cuh, grad_tile_kernel) to autograd so the O(p) chain rule to the raw parameters and the
    prior terms stay ordinary torch code (optim/mll_scipy.py:37-60, :112-127)."""

    @staticmethod
    def forward(ctx, model, w, z, sf2, noise, beta):
        eng = model._get_engine()
        hyper = {"w": w.detach().double().cpu().numpy(),
                 "z": z.detach().double().cpu().numpy() if eng.dz > 0 else None,
                 "sigma_f2": float(sf2.detach()),
                 "noise": noise.detach().double().cpu().numpy().reshape(-1),
                 "beta": beta.detach().double().cpu().numpy().reshape(-1) if eng.n_mean > 0 else None}
        need_grad = any(ctx.needs_input_grad[1:])
        out = eng.mll_grad(hyper, want_grad=need_grad)
        model._last_eval = out
        model._factor_key = None  # the engine's factor now belongs to these hyper-parameters (no prediction cache)
        if need_grad:
            ctx.grads = (
                torch.as_tensor(-out["d_w"], dtype=w.dtype).reshape(w.shape),
                torch.as_tensor(-out["d_z"], dtype=z.dtype).reshape(z.shape) if eng.dz > 0 else torch.zeros_like(z),
                torch.as_tensor(-out["d_sigma_f2"], dtype=sf2.dtype).reshape(sf2.shape),
                torch.as_tensor(-out["d_noise"], dtype=noise.dtype).reshape(noise.shape),
                torch.as_tensor(-out["d_beta"], dtype=beta.dtype).reshape(beta.shape) if eng.n_mean > 0
                else torch.zeros_like(beta),
            )
        return torch.tensor(-out["nll"], dtype=torch.float64)

    @staticmethod
    def backward(ctx, g):
        gw, gz, gs, gn, gb = ctx.grads
        g = g.to(torch.float64)
        return (None, (g * gw).to(gw.dtype), (g * gz).to(gz.dtype), (g * gs).to(gs.dtype), (g * gn).to(gn.dtype),
                (g * gb).to(gb.dtype))


class _EnginePrediction(torch.autograd.Function):
    """Scaled predictive mean and clamped variance at the rows of ``x`` (gpp_predict_grad), differentiable w.r.t. the
    quantitative columns of ``x``: the graph the reference's ``GPR.predict`` keeps when its inputs require a gradient
    (models/gpregression.py:122-149, reached through GP_Plus.predict_with_grad, models/gp_plus.py:626-628).
    Categorical and source columns get a zero gradient (the reference turns them into integer indices), the
    hyper-parameters none.  First derivatives only: differentiating the backward raises."""

    @staticmethod
    def forward(ctx, x, eng, xq, cols, kwargs):
        mean, var, d_mean, d_var = eng.predict_grad(xq, **kwargs)
        mean, var = torch.from_numpy(np.asarray(mean)), torch.from_numpy(np.asarray(var))
        ctx.x_meta = (x.shape, x.dtype, x.device)
        ctx.cols = cols
        ctx.d_mean = torch.as_tensor(np.asarray(d_mean), dtype=torch.float64).reshape(len(mean), len(cols))
        # a variance at min_var was clamped there: no gradient, as through torch's clamp_min
        d_var = torch.as_tensor(np.asarray(d_var), dtype=torch.float64).reshape(len(var), len(cols))
        ctx.d_var = torch.where((var > kwargs["min_var"])[:, None], d_var, torch.zeros_like(d_var))
        return mean, var

    @staticmethod
    @once_differentiable
    def backward(ctx, g_mean, g_var):
        shape, dtype, device = ctx.x_meta
        gq = g_mean.double()[:, None] * ctx.d_mean + g_var.double()[:, None] * ctx.d_var
        gx = torch.zeros(shape, dtype=dtype, device=device)
        gx[:, ctx.cols] = gq.to(dtype=dtype, device=device)
        return gx, None, None, None, None


class _EngineQBatchPosterior(torch.autograd.Function):
    """Scaled means [b, q] and joint covariances [b, q, q] of b t-batches of q consecutive rows of ``x``
    (gpp_posterior_qbatch), differentiable w.r.t. the quantitative columns of ``x``: the backward runs
    gpp_posterior_qbatch_grad at the same rows with the hyper-parameters of the forward.  Categorical and source
    columns get a zero gradient, the hyper-parameters none.  First derivatives only: differentiating the backward
    raises."""

    @staticmethod
    def forward(ctx, x, model, eng, xq, q, kwargs):
        mean, cov = eng.posterior_qbatch(xq, q, **kwargs)
        ctx.set_materialize_grads(False)
        ctx.x_meta = (x.shape, x.dtype, x.device)
        ctx.request = (model, eng, model._factor_key, model._hyper_numpy(), xq, q, kwargs)
        return torch.from_numpy(np.asarray(mean)), torch.from_numpy(np.asarray(cov))

    @staticmethod
    @once_differentiable
    def backward(ctx, g_mean, g_cov):
        shape, dtype, device = ctx.x_meta
        model, eng, key, hyper, xq, q, kwargs = ctx.request
        gx = torch.zeros(shape, dtype=dtype, device=device)
        cols = model._quant_columns()
        if len(cols) == 0 or (g_mean is None and g_cov is None):
            return gx, None, None, None, None, None
        if model._factor_key != key:  # the engine was refactorised since the forward: restore its hyper-parameters
            eng.factorize(hyper)
            model._factor_key = key
            model._ipv_state = None
        gm, gc = (None if g is None else np.ascontiguousarray(g.detach().double().cpu().numpy()) for g in (g_mean, g_cov))
        d_xq = eng.posterior_qbatch_grad(xq, q, gm, gc, **kwargs)
        gx[:, cols] = torch.as_tensor(np.asarray(d_xq), dtype=torch.float64).reshape(-1, len(cols)).to(dtype=dtype,
                                                                                                     device=device)
        return gx, None, None, None, None, None


_QACQ_KINDS = {"qEI": _engine.QACQ_EI, "qNEI": _engine.QACQ_NEI, "qUCB": _engine.QACQ_UCB}


def sobol_normal_samples(num_samples: int, dim: int, seed: int = 0) -> torch.Tensor:
    """[num_samples, dim] scrambled Sobol points mapped through the normal inverse CDF (botorch's
    ``draw_sobol_normal_samples``, the base samples of ``SobolQMCNormalSampler``)."""
    u = torch.quasirandom.SobolEngine(dimension=int(dim), scramble=True, seed=int(seed)).draw(int(num_samples),
                                                                                            dtype=torch.float64)
    v = 0.5 + (1.0 - torch.finfo(u.dtype).eps) * (u - 0.5)
    return torch.erfinv(2.0 * v - 1.0) * math.sqrt(2.0)


class _EngineQBatchAcquisition(torch.autograd.Function):
    """Monte-Carlo batch acquisition values [b] of the t-batches of ``x`` [b, q, d] (gpp_acq_qbatch), differentiable
    w.r.t. the quantitative columns of ``x``: the forward asks the engine for d(sum values)/dx as well, and the backward
    scales each t-batch's rows by its upstream gradient.  Categorical and source columns get a zero gradient, the
    baseline rows and the hyper-parameters none.  First derivatives only: differentiating the backward raises."""

    @staticmethod
    def forward(ctx, x, eng, xq, q_tot, cols, kwargs):
        values, d_xq, jitter = eng.acquisition_qbatch(xq, q_tot, want_grad=len(cols) > 0, **kwargs)
        b, q, d = x.shape
        dx = torch.zeros(b, q, d, dtype=torch.float64)
        if len(cols) > 0:
            dx[:, :, cols] = torch.as_tensor(np.asarray(d_xq)).reshape(b, q_tot, len(cols))[:, :q]
        ctx.dx = dx
        ctx.x_meta = (x.dtype, x.device)
        jitter = torch.as_tensor(np.asarray(jitter))
        ctx.mark_non_differentiable(jitter)
        return torch.as_tensor(np.asarray(values)), jitter

    @staticmethod
    @once_differentiable
    def backward(ctx, g_values, g_jitter):
        dtype, device = ctx.x_meta
        if g_values is None:
            return (torch.zeros(ctx.dx.shape, dtype=dtype, device=device),) + (None,) * 5
        gx = g_values.double().reshape(-1, 1, 1).cpu() * ctx.dx
        return (gx.to(dtype=dtype, device=device),) + (None,) * 5


class _EngineNIPV(_EngineQBatchAcquisition):
    """Negative integrated posterior variances [b] of the t-batches of ``x`` [b, q, d] against the engine's stored
    integration set (gpp_nipv_qbatch), differentiable w.r.t. the quantitative columns of ``x`` as
    ``_EngineQBatchAcquisition``, whose backward it shares."""

    @staticmethod
    def forward(ctx, x, eng, xq, q, cols, kwargs):
        values, d_xq, jitter = eng.nipv_qbatch(xq, q, want_grad=len(cols) > 0, **kwargs)
        b, _, d = x.shape
        dx = torch.zeros(b, q, d, dtype=torch.float64)
        if len(cols) > 0:
            dx[:, :, cols] = torch.as_tensor(np.asarray(d_xq)).reshape(b, q, len(cols))
        ctx.dx = dx
        ctx.x_meta = (x.dtype, x.device)
        jitter = torch.as_tensor(np.asarray(jitter))
        ctx.mark_non_differentiable(jitter)
        return torch.as_tensor(np.asarray(values)), jitter


class _EngineKG(_EngineQBatchAcquisition):
    """One-shot knowledge-gradient values [b] of the t-batches of ``x`` [b, q + F, d] (gpp_kg_qbatch), differentiable
    w.r.t. the quantitative columns of all q + F rows as ``_EngineQBatchAcquisition``, whose backward it shares."""

    @staticmethod
    def forward(ctx, x, eng, xq, q, cols, kwargs):
        b, q_tot, d = x.shape
        values, d_xq, jitter = eng.kg_qbatch(xq, q, q_tot - q, want_grad=len(cols) > 0, **kwargs)
        dx = torch.zeros(b, q_tot, d, dtype=torch.float64)
        if len(cols) > 0:
            dx[:, :, cols] = torch.as_tensor(np.asarray(d_xq)).reshape(b, q_tot, len(cols))
        ctx.dx = dx
        ctx.x_meta = (x.dtype, x.device)
        jitter = torch.as_tensor(np.asarray(jitter))
        ctx.mark_non_differentiable(jitter)
        return torch.as_tensor(np.asarray(values)), jitter


class _EngineGIBBON(_EngineQBatchAcquisition):
    """GIBBON values [b] of the t-batches of ``x`` [b, q, d] (gpp_gibbon_qbatch), differentiable w.r.t. the
    quantitative columns of ``x`` as ``_EngineQBatchAcquisition``, whose backward it shares.  The engine's t-batches
    hold the q rows of ``x``, then the pending rows, then (projected) the target copies of both.  ``layout`` is
    (q_eff, held): q_eff rows per half, and the columns the target rows hold at a fixed value.  A target row copies
    every other quantitative column of its actual row, so row i's gradient in column c is d_xq[i, c] +
    d_xq[q_eff + i, c], and d_xq[i, c] alone for a held column.  Pending rows get none."""

    @staticmethod
    def forward(ctx, x, eng, xq, layout, cols, kwargs):
        b, q, d = x.shape
        q_eff, held = layout
        values, d_xq, jitter = eng.gibbon_qbatch(xq, q_eff, want_grad=len(cols) > 0, **kwargs)
        dx = torch.zeros(b, q, d, dtype=torch.float64)
        if len(cols) > 0:
            g = torch.as_tensor(np.asarray(d_xq)).reshape(b, -1, len(cols))
            if kwargs["projected"]:
                copied = torch.tensor([c not in held for c in cols], dtype=torch.float64)
                g = g[:, :q_eff] + g[:, q_eff:] * copied
            dx[:, :, cols] = g[:, :q]
        ctx.dx = dx
        ctx.x_meta = (x.dtype, x.device)
        jitter = torch.as_tensor(np.asarray(jitter))
        ctx.mark_non_differentiable(jitter)
        return torch.as_tensor(np.asarray(values)), jitter


class GPR(Module):
    def __init__(
        self,
        train_x: torch.Tensor,
        train_y: torch.Tensor,
        correlation_kernel,
        noise_indices: List[int],
        fix_noise: bool = False,
        fix_noise_val: float = 1e-5,
        lb_noise: float = 1e-12,
    ) -> None:
        if not torch.is_tensor(train_x):
            raise RuntimeError("'train_x' must be a tensor")
        if not torch.is_tensor(train_y):
            raise RuntimeError("'train_y' must be a tensor")
        if train_x.shape[0] != train_y.shape[0]:
            raise RuntimeError("Inputs and output have different number of observations")
        super().__init__()

        noise_constraint = GreaterThan(lb_noise, transform=torch.exp, inv_transform=torch.log)
        if len(noise_indices) == 0:
            likelihood = GaussianLikelihood(noise_constraint=noise_constraint)
        else:
            likelihood = Multifidelity_likelihood(noise_constraint=noise_constraint, noise_indices=noise_indices,
                                                  fidel_indices=train_x[:, -1])
        y_min = train_y.min()
        y_std = train_y.max() - train_y.min()
        train_y_sc = (train_y - y_min) / y_std

        self.train_inputs = (train_x,)
        self.train_targets = train_y_sc
        self.likelihood = likelihood
        self.register_buffer("y_min", y_min)
        self.register_buffer("y_std", y_std)
        self.register_buffer("y_scaled", train_y_sc)
        self._num_outputs = 1

        self.likelihood.register_prior("noise_prior", LogHalfHorseshoePrior(0.01, lb_noise), "raw_noise")
        if fix_noise:
            self.likelihood.raw_noise.requires_grad_(False)
            self.likelihood.noise_covar.noise = torch.tensor(fix_noise_val)

        if isinstance(correlation_kernel, str):
            try:
                kernel_class = getattr(kernels, correlation_kernel)
                correlation_kernel = kernel_class(
                    ard_num_dims=self.train_inputs[0].size(1),
                    lengthscale_constraint=Positive(transform=torch.exp, inv_transform=torch.log),
                )
                correlation_kernel.register_prior(
                    "lengthscale_prior", MollifiedUniformPrior(math.log(0.1), math.log(10)), "raw_lengthscale")
            except Exception:
                raise RuntimeError("%s not an allowed kernel" % correlation_kernel)
        elif not isinstance(correlation_kernel, Kernel):
            raise RuntimeError("specified correlation kernel is not a `gpytorch.kernels.Kernel` instance")

        self.covar_module = kernels.ScaleKernel(
            base_kernel=correlation_kernel,
            outputscale_constraint=Positive(transform=softplus, inv_transform=inv_softplus),
        )
        self.covar_module.register_prior("outputscale_prior", LogNormalPrior(1e-6, 1.0), "outputscale")

        # engine state (never pickled / deep-copied)
        self._engine = None
        self._engine_device = None
        self._factor_key = None
        self._last_eval = None
        self._ipv_state = None  # (engine, factor key, integration inputs, levels) of the engine's qNIPV set

    # ------------------------------------------------------------------------------------------
    # engine plumbing
    def __getstate__(self):
        state = self.__dict__.copy()
        state["_engine"] = None
        state["_factor_key"] = None
        state["_last_eval"] = None
        state["_ipv_state"] = None
        return state

    def __deepcopy__(self, memo):
        import copy
        cls = self.__class__
        new = cls.__new__(cls)
        memo[id(self)] = new
        for k, v in self.__dict__.items():
            if k in ("_engine", "_last_eval", "_ipv_state"):
                new.__dict__[k] = None
            elif k == "_factor_key":
                new.__dict__[k] = None
            else:
                new.__dict__[k] = copy.deepcopy(v, memo)
        return new

    def _quant_columns(self) -> List[int]:
        return list(range(self.train_inputs[0].shape[-1]))

    def _level_index(self, x: torch.Tensor, training: bool) -> Optional[np.ndarray]:
        return None

    def _latent_table(self) -> Optional[torch.Tensor]:
        return None

    def _latent_passes(self) -> int:
        return 1

    def _check_combos_seen(self, levels):
        return None

    def _quant_kernel(self):
        leaves = [k for k in self.covar_module.leaf_kernels() if k.has_lengthscale]
        if len(leaves) != 1:
            raise RuntimeError("GPR expects exactly one stationary kernel under ScaleKernel")
        return leaves[0]

    def _noise_index(self, x: torch.Tensor) -> Optional[np.ndarray]:
        if isinstance(self.likelihood, Multifidelity_likelihood):
            return self.likelihood.group_index(x[:, -1]).numpy()
        return None

    def _mean_layout(self) -> Tuple[int, List[torch.nn.Parameter]]:
        """(n_mean, constants) of the mean model: ZeroMean -> 0, ConstantMean -> 1."""
        mm = getattr(self, "mean_module", None)
        if mm is None or isinstance(mm, ZeroMean):
            return 0, []
        if isinstance(mm, ConstantMean):
            return 1, [mm.constant]
        raise NotImplementedError("mean module %s has no device path" % type(mm).__name__)

    def _mean_index(self, x: torch.Tensor) -> Optional[np.ndarray]:
        return None

    def _engine_kwargs(self, dev: int) -> dict:
        """Constructor arguments of an engine handle holding this model's training set on GPU ``dev``."""
        x = self.train_inputs[0]
        qk = self._quant_kernel() if len(self._quant_columns()) > 0 else None
        family = qk.family if qk is not None else _engine.KERNEL_EXPSQ
        with torch.no_grad():
            table = self._latent_table()
        n_mean, _ = self._mean_layout()
        n_noise = int(self.likelihood.noise_covar.raw_noise.numel())
        xq = x[:, self._quant_columns()].detach().double().cpu().numpy() if qk is not None else None
        return dict(
            xq=xq, y=self.train_targets.detach().double().cpu().numpy(), kernel=family,
            level_idx=self._level_index(x, True), n_combo=0 if table is None else int(table.shape[-2]),
            dz=0 if table is None else int(table.shape[-1]), noise_idx=self._noise_index(x), n_noise=n_noise,
            mean_idx=self._mean_index(x), n_mean=n_mean, device=dev, n_pass=self._latent_passes())

    def _new_engine(self, dev: int, kwargs: Optional[dict] = None) -> "_engine.Engine":
        """A fresh engine handle holding this model's training set on GPU ``dev`` (not cached: the lock-step
        multi-start driver keeps one handle per in-flight restart and passes the same ``kwargs`` to all of them)."""
        return _engine.Engine(**(kwargs if kwargs is not None else self._engine_kwargs(dev)))

    @contextlib.contextmanager
    def engine_override(self, engine):
        """Route every engine call of this model to ``engine`` inside the block (the closed-form objective is validated
        against the torch path through a stub engine, optim/_fast_objective.self_check); the real engine, its
        factorisation cache and the parameters are untouched."""
        prev = getattr(self, "_engine_stub", None)
        self._engine_stub = engine
        try:
            yield engine
        finally:
            self._engine_stub = prev
            self._factor_key = None

    def _get_engine(self) -> "_engine.Engine":
        if getattr(self, "_engine_stub", None) is not None:
            return self._engine_stub
        dev = get_default_device()
        if self._engine is not None and self._engine_device == dev and self._engine.n_pass == self._latent_passes():
            return self._engine
        if self._engine is not None:
            self._engine.close()
        self._engine = self._new_engine(dev)
        self._engine_device = dev
        self._factor_key = None
        return self._engine

    def release_engine(self):
        if self._engine is not None:
            self._engine.close()
        self._engine = None
        self._factor_key = None

    def _natural(self):
        """Differentiable natural hyper-parameters (w, Z, sigma_f^2, noise, beta) from the raw ones."""
        ref = self.covar_module.raw_outputscale
        if len(self._quant_columns()) > 0:
            w = self._quant_kernel().distance_weights()
        else:
            w = torch.zeros(0, dtype=ref.dtype)
        z = self._latent_table()
        if z is None:
            z = torch.zeros(0, dtype=ref.dtype)
        sf2 = self.covar_module.outputscale
        noise = self.likelihood.noise.reshape(-1)
        n_mean, consts = self._mean_layout()
        beta = torch.cat([c.reshape(-1) for c in consts]) if n_mean > 0 else torch.zeros(0, dtype=ref.dtype)
        return w, z, sf2, noise, beta

    def log_marginal(self) -> torch.Tensor:
        """log p(y_scaled | X, theta): differentiable float64 scalar, NOT divided by n."""
        w, z, sf2, noise, beta = self._natural()
        return _EngineLogProb.apply(self, w, z, sf2, noise, beta)

    def prior_mean_and_variance(self):
        """Prior mean vector and prior variance (diag of sigma_f^2 * correlation = sigma_f^2) at the training inputs
        as differentiable float64 tensors -- what ``model(*model.train_inputs)`` returns in training mode
        (gp_plus.py:386-484); used by the interval-score penalty (mll_scipy.py:57-59)."""
        x = self.train_inputs[0]
        n = x.shape[0]
        n_mean, consts = self._mean_layout()
        if n_mean == 0:
            mean = torch.zeros(n, dtype=torch.float64)
        else:
            beta = torch.cat([c.reshape(-1) for c in consts]).to(torch.float64)
            idx = self._mean_index(x)
            if idx is None:
                mean = beta[0].expand(n)
            else:
                idx = torch.as_tensor(idx, dtype=torch.long)
                mean = torch.where(idx >= 0, beta[idx.clamp_min(0)], torch.zeros(n, dtype=torch.float64))
        var = self.covar_module.outputscale.to(torch.float64).reshape(()).expand(n)
        return mean, var

    def _hyper_numpy(self):
        with torch.no_grad():
            w, z, sf2, noise, beta = self._natural()
        eng = self._get_engine()
        return {"w": w.double().numpy(), "z": z.double().numpy() if eng.dz > 0 else None, "sigma_f2": float(sf2),
                "noise": noise.double().numpy(), "beta": beta.double().numpy() if eng.n_mean > 0 else None}

    def _ensure_factor(self):
        eng = self._get_engine()
        hyper = self._hyper_numpy()
        key = tuple(np.concatenate([np.ravel(v) for v in (hyper["w"], hyper["z"] if hyper["z"] is not None else [],
                                                           [hyper["sigma_f2"]], hyper["noise"],
                                                           hyper["beta"] if hyper["beta"] is not None else [])]).tolist())
        if self._factor_key != key:
            eng.factorize(hyper)
            self._factor_key = key
            self._ipv_state = None  # the engine drops its integration set with the old factor
        return eng

    # ------------------------------------------------------------------------------------------
    def forward(self, x: torch.Tensor) -> MultivariateNormal:
        """Prior mean and dense covariance at x (off the hot path; kept for API compatibility)."""
        mm = getattr(self, "mean_module", None)
        mean_x = mm(x) if mm is not None else torch.zeros(x.shape[0], dtype=x.dtype)
        covar_x = self.covar_module.outputscale * self.covar_module.base_kernel(x).evaluate()
        return MultivariateNormal(mean_x, covar_x)

    def predict(self, x: torch.Tensor, return_std: bool = False, include_noise: bool = False
                ) -> Union[torch.Tensor, Tuple[torch.Tensor]]:
        """Posterior mean (and standard deviation) in the original y units (gpregression.py:122-149).

        When gradients are enabled and ``x`` requires one, the outputs carry a graph back to the quantitative columns
        of ``x`` (gpp_predict_grad; the values are bitwise those of the plain call); otherwise they carry none."""
        self.eval()
        with settings.fast_computations(log_prob=False):
            if self.train_targets.ndim != 1:
                raise NotImplementedError("batched GPs are not supported by the engine")
            if x.dim() != 2:
                raise ValueError("predict expects a 2-D tensor of inputs")
            eng = self._ensure_factor()
            self.fidel_indices = x[:, -1]
            xc = x.detach().cpu()
            cols = self._quant_columns()
            xq = xc[:, cols].double().numpy() if len(cols) > 0 else np.zeros((xc.shape[0], 0))
            add_noise = bool(return_std and include_noise)
            if add_noise and isinstance(self.likelihood, Multifidelity_likelihood):
                self.likelihood.fidel_indices = x[:, -1]
            levels = self._level_index(xc, False)
            if levels is not None:
                self._check_combos_seen(levels)
            kwargs = dict(level_idx=levels, noise_idx=self._noise_index(xc) if add_noise else None,
                          mean_idx=self._mean_index(xc), include_noise=add_noise, min_var=settings.min_variance)
            if torch.is_grad_enabled() and x.requires_grad:
                mean_sc, var_sc = _EnginePrediction.apply(x, eng, np.ascontiguousarray(xq), cols, kwargs)
            else:
                mean_sc, var_sc = (torch.from_numpy(a) for a in eng.predict(np.ascontiguousarray(xq), **kwargs))
            dtype = self.y_std.dtype if self.y_std.dtype.is_floating_point else torch.float64
            out_mean = self.y_min + self.y_std * mean_sc.to(dtype)
            if return_std:
                out_std = var_sc.to(dtype).sqrt() * self.y_std
                return out_mean, out_std
            return out_mean

    def _joint_request(self, x: torch.Tensor, include_noise: bool):
        """Engine (factorised for the current hyper-parameters), quantitative inputs and index arguments of a joint
        posterior call at the rows of ``x``: levels, noise groups and means exactly as ``predict`` gathers them."""
        self.eval()
        if self.train_targets.ndim != 1:
            raise NotImplementedError("batched GPs are not supported by the engine")
        if x.dim() != 2:
            raise ValueError("expected a 2-D tensor of inputs")
        eng = self._ensure_factor()
        xc = x.detach().cpu()
        cols = self._quant_columns()
        xq = xc[:, cols].double().numpy() if len(cols) > 0 else np.zeros((xc.shape[0], 0))
        levels = self._level_index(xc, False)
        if levels is not None:
            self._check_combos_seen(levels)
        kwargs = dict(level_idx=levels, noise_idx=self._noise_index(xc) if include_noise else None,
                      mean_idx=self._mean_index(xc), include_noise=bool(include_noise))
        return eng, np.ascontiguousarray(xq), kwargs

    def _out_dtype(self):
        return self.y_std.dtype if self.y_std.dtype.is_floating_point else torch.float64

    def predict_joint(self, x: torch.Tensor, include_noise: bool = False) -> Tuple[torch.Tensor, torch.Tensor]:
        """Posterior mean [M] and full covariance [M, M] at the rows of ``x`` in the original y units: the joint
        structure that the reference's ``posterior`` carries (gpregression.py:151-166).  The mean equals ``predict``'s;
        the covariance is exactly symmetric and not clamped.  ``include_noise`` adds each row's observation noise on
        the diagonal.  No autograd graph; M is at most ``_engine.MAX_JOINT``."""
        with torch.no_grad():
            eng, xq, kwargs = self._joint_request(x, include_noise)
            mean_sc, cov_sc = eng.predict_joint(xq, **kwargs)
            dtype = self._out_dtype()
            mean = self.y_min + self.y_std * torch.as_tensor(np.asarray(mean_sc)).to(dtype)
            cov = (self.y_std * self.y_std) * torch.as_tensor(np.asarray(cov_sc)).to(dtype)
        return mean, cov

    def sample_posterior(self, x: torch.Tensor, num_samples: int = 1, include_noise: bool = False,
                         base_samples: Optional[torch.Tensor] = None, generator: Optional[torch.Generator] = None
                         ) -> torch.Tensor:
        """``num_samples`` draws [S, M] from the joint posterior at the rows of ``x``, in the original y units
        (gpytorch ``MultivariateNormal.rsample``): ``mean + base_samples L^T`` with ``L`` the Cholesky factor of the
        posterior covariance.  The default base samples are ``torch.randn(S, M, generator=generator)`` in float64 on
        the CPU, as gpytorch draws them; a singular covariance gets the psd_safe_cholesky jitter and a warning."""
        with torch.no_grad():
            eng, xq, kwargs = self._joint_request(x, include_noise)
            m = xq.shape[0]
            if base_samples is None:
                base_samples = torch.randn(int(num_samples), m, generator=generator, dtype=torch.float64)
            else:
                base_samples = torch.as_tensor(base_samples)
            if tuple(base_samples.shape) != (int(num_samples), m):
                raise ValueError("base_samples must have shape %s, got %s"
                                 % ((int(num_samples), m), tuple(base_samples.shape)))
            base = np.ascontiguousarray(base_samples.detach().to(device="cpu", dtype=torch.float64).numpy())
            samples_sc, jitter = eng.sample_posterior(xq, base, **kwargs)
            if jitter > 0:
                warnings.warn("A not p.d., added jitter of %.1e to the diagonal" % jitter, NumericalWarning)
            dtype = self._out_dtype()
            return self.y_min + self.y_std * torch.as_tensor(np.asarray(samples_sc)).to(dtype)

    def posterior(self, X, output_indices=None, observation_noise=True, posterior_transform=None, **kwargs):
        """Predictive distribution at X in SCALED units (botorch posterior stand-in); differentiable in X when X
        requires a gradient.  A 2-D X [m, d] gives the mean and the marginal variances (GPR.predict, which subclasses'
        no_grad predict wraps).  X [..., q, d] gives the joint distribution of every t-batch of q points, mean
        [..., q] and covariance [..., q, q], the input of Monte-Carlo batch acquisition (qEI, qNEI, qUCB, qKG)."""
        self.eval()
        X = X.double()
        if X.dim() >= 3:
            return self._posterior_qbatch(X, bool(observation_noise))
        mean, std = GPR.predict(self, X, return_std=True, include_noise=bool(observation_noise))
        mu = (mean - self.y_min) / self.y_std
        var = (std / self.y_std) ** 2
        return MultivariateNormal(mu, torch.diag(var))

    def _posterior_qbatch(self, X: torch.Tensor, include_noise: bool) -> MultivariateNormal:
        """Joint posterior of the t-batches of X [..., q, d] (gpp_posterior_qbatch): the leading dimensions are
        flattened into b t-batches, whose rows are gathered as ``predict`` gathers one 2-D batch (categorical columns
        ranked against the training inputs and all rows of X)."""
        batch, q = X.shape[:-2], int(X.shape[-2])
        x = X.reshape(-1, X.shape[-1])
        eng, xq, kwargs = self._joint_request(x, include_noise)
        if torch.is_grad_enabled() and X.requires_grad:
            mean, cov = _EngineQBatchPosterior.apply(x, self, eng, xq, q, kwargs)
        else:
            mean, cov = (torch.from_numpy(np.asarray(a)) for a in eng.posterior_qbatch(xq, q, **kwargs))
        return MultivariateNormal(mean.reshape(*batch, q), cov.reshape(*batch, q, q))

    def acquisition_qbatch(self, X: torch.Tensor, kind: str = "qEI", best_f: Optional[float] = None,
                           X_baseline: Optional[torch.Tensor] = None, beta: Optional[float] = None,
                           num_samples: int = 512, base_samples: Optional[torch.Tensor] = None, seed: int = 0,
                           maximize: bool = True, observation_noise: bool = False,
                           mc_points: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Monte-Carlo batch acquisition (botorch's qEI, qNEI, qUCB) of every t-batch of X [..., q, d], in the original
        y units: values [...] (gpp_acq_qbatch).  All t-batches share the base samples [S, q + n_b], by default
        ``num_samples`` scrambled Sobol normal draws of ``seed`` (botorch's SobolQMCNormalSampler), so each value is a
        deterministic function of its own t-batch and L-BFGS-B can optimise it.  qEI needs ``best_f``, qNEI the
        baseline points ``X_baseline`` [n_b, d] appended to every t-batch (q + n_b <= 128), qUCB ``beta``.  The values
        are differentiable in the quantitative columns of X when X requires a gradient; a t-batch whose covariance
        needed jitter raises a NumericalWarning.

        ``kind="qNIPV"`` (botorch's qNegIntegratedPosteriorVariance) needs ``mc_points`` [M, d], the integration
        points, and takes none of ``best_f``, ``beta``, ``X_baseline`` or ``base_samples``: the value is minus the mean,
        over ``mc_points``, of the latent posterior variance after also observing the t-batch with its observation
        noise, in y units squared.  It is exact (no samples), and the source column of ``mc_points`` selects which
        fidelity's variance is integrated."""
        if kind == "qNIPV":
            given = [k for k, v in (("best_f", best_f), ("beta", beta), ("X_baseline", X_baseline),
                                    ("base_samples", base_samples)) if v is not None]
            if given:
                raise ValueError("acquisition_qbatch: qNIPV takes no %s" % ", ".join(given))
            if mc_points is None:
                raise ValueError("acquisition_qbatch: qNIPV needs mc_points")
            return self._nipv_qbatch(X, mc_points)
        if mc_points is not None:
            raise ValueError("acquisition_qbatch: mc_points is for qNIPV only")
        if kind not in _QACQ_KINDS:
            raise ValueError("acquisition_qbatch: kind must be one of %s, got %r"
                             % (sorted(list(_QACQ_KINDS) + ["qNIPV"]), kind))
        if kind == "qEI" and best_f is None:
            raise ValueError("acquisition_qbatch: qEI needs best_f")
        if kind == "qNEI" and X_baseline is None:
            raise ValueError("acquisition_qbatch: qNEI needs X_baseline")
        if kind == "qUCB" and beta is None:
            raise ValueError("acquisition_qbatch: qUCB needs beta")
        if X.dim() < 2:
            raise ValueError("acquisition_qbatch expects X of shape [..., q, d]")
        self.eval()
        batch, q, d = X.shape[:-2], int(X.shape[-2]), int(X.shape[-1])
        x = X.reshape(-1, q, d)
        b = x.shape[0]
        n_b = 0
        rows = x.detach().double()
        if kind == "qNEI":
            Xb = torch.as_tensor(X_baseline).detach().double().reshape(-1, d)
            n_b = Xb.shape[0]
            if n_b < 1:
                raise ValueError("acquisition_qbatch: X_baseline has no rows")
            rows = torch.cat([rows, Xb.to(rows.device).expand(b, n_b, d)], dim=1)
        q_tot = q + n_b
        if q_tot > _engine.MAX_QBATCH:
            raise ValueError("acquisition_qbatch: q + n_baseline = %d exceeds %d" % (q_tot, _engine.MAX_QBATCH))
        if base_samples is None:
            base_samples = sobol_normal_samples(num_samples, q_tot, seed)
        base = np.ascontiguousarray(torch.as_tensor(base_samples).detach().to("cpu", torch.float64).numpy())
        if base.ndim != 2 or base.shape[1] != q_tot:
            raise ValueError("acquisition_qbatch: base_samples must have shape [S, %d], got %s" % (q_tot, base.shape))
        y_min, y_std = float(self.y_min), float(self.y_std)
        sgn = 1.0 if maximize else -1.0
        eng, xq, kwargs = self._joint_request(rows.reshape(-1, d), bool(observation_noise))
        kwargs.update(kind=_QACQ_KINDS[kind], base_samples=base, n_baseline=n_b, maximize=bool(maximize),
                      best_f=0.0 if best_f is None else (float(best_f) - y_min) / y_std,
                      beta=0.0 if beta is None else float(beta))
        if torch.is_grad_enabled() and X.requires_grad:
            v, jitter = _EngineQBatchAcquisition.apply(x, eng, xq, q_tot, self._quant_columns(), kwargs)
        else:
            values, _, jitter = eng.acquisition_qbatch(xq, q_tot, want_grad=False, **kwargs)
            v, jitter = torch.as_tensor(np.asarray(values)), torch.as_tensor(np.asarray(jitter))
        if bool((jitter > 0).any()):
            warnings.warn("A not p.d., added jitter of %.1e to the diagonal" % float(jitter.max()), NumericalWarning)
        dtype = self._out_dtype()
        v = v.to(dtype)
        out = sgn * y_min + y_std * v if kind == "qUCB" else y_std * v
        return out.reshape(batch)

    def _nipv_qbatch(self, X: torch.Tensor, mc_points) -> torch.Tensor:
        if X.dim() < 2:
            raise ValueError("acquisition_qbatch expects X of shape [..., q, d]")
        self.eval()
        batch, q, d = X.shape[:-2], int(X.shape[-2]), int(X.shape[-1])
        if q > _engine.MAX_QBATCH:
            raise ValueError("acquisition_qbatch: q = %d exceeds %d" % (q, _engine.MAX_QBATCH))
        x = X.reshape(-1, q, d)
        n_c = x.shape[0] * q
        P = torch.as_tensor(mc_points).detach().double()
        if P.dim() != 2 or P.shape[1] != d:
            raise ValueError("acquisition_qbatch: mc_points must have shape [M, %d], got %s" % (d, tuple(P.shape)))
        if not 1 <= P.shape[0] <= _engine.MAX_IPV_POINTS:
            raise ValueError("acquisition_qbatch: mc_points must have 1 to %d rows" % _engine.MAX_IPV_POINTS)
        # candidates and integration points are ranked together against the training inputs, as qNEI's baseline
        rows = torch.cat([x.detach().double().reshape(-1, d), P.to(x.device)])
        eng, xq, kw = self._joint_request(rows, True)
        lv, nz = kw["level_idx"], kw["noise_idx"]
        xq_i = np.ascontiguousarray(xq[n_c:])
        lv_i = None if lv is None else np.ascontiguousarray(lv[n_c:])
        st = self._ipv_state
        if not (st is not None and st[0] is eng and st[1] == self._factor_key and np.array_equal(st[2], xq_i)
                and (st[3] is None if lv_i is None else (st[3] is not None and np.array_equal(st[3], lv_i)))):
            self._ipv_state = None
            eng.ipv_points(xq_i, level_idx=lv_i)
            self._ipv_state = (eng, self._factor_key, xq_i, lv_i)
        kwargs = dict(level_idx=None if lv is None else np.ascontiguousarray(lv[:n_c]),
                      noise_idx=None if nz is None else np.ascontiguousarray(nz[:n_c]))
        xq_c = np.ascontiguousarray(xq[:n_c])
        if torch.is_grad_enabled() and X.requires_grad:
            v, jitter = _EngineNIPV.apply(x, eng, xq_c, q, self._quant_columns(), kwargs)
        else:
            values, _, jitter = eng.nipv_qbatch(xq_c, q, want_grad=False, **kwargs)
            v, jitter = torch.as_tensor(np.asarray(values)), torch.as_tensor(np.asarray(jitter))
        if bool((jitter > 0).any()):
            warnings.warn("A not p.d., added jitter of %.1e to the diagonal" % float(jitter.max()), NumericalWarning)
        y_std = self.y_std.to(self._out_dtype())
        return (y_std * y_std * v.to(self._out_dtype())).reshape(batch)

    def knowledge_gradient(self, X: torch.Tensor, num_fantasies: int, base_samples: Optional[torch.Tensor] = None,
                           seed: int = 0, maximize: bool = True, current_value: Optional[float] = None,
                           cost_by_source=None) -> torch.Tensor:
        """One-shot knowledge gradient (botorch's qKnowledgeGradient with the PosteriorMean value function) of every
        t-batch of X [..., q + F, d] in the original y units: values [...] (gpp_kg_qbatch).  The last F =
        ``num_fantasies`` rows of each t-batch are the fantasy solutions and the first q the actual points (botorch's
        X_actual_and_fantasies).  The value is the mean over the fantasies f of sigma times the posterior mean at
        fantasy solution f after also observing the actual points, each with its observation noise, at y_f = mu + L
        e_f (sigma = +1 to maximise, -1 to minimise).  All t-batches share the base samples e [F, q], by default
        ``num_fantasies`` scrambled Sobol normal draws of ``seed``.

        ``current_value`` (original units, times sigma like the values: the best posterior mean, e.g. from
        ``optimize_posterior_mean``) is subtracted.  ``cost_by_source`` ({source: cost} or a sequence indexed by
        source; needs ``current_value``) then divides that gain by the summed cost of the q actual rows, whose source
        is the last column of X: botorch's qMultiFidelityKnowledgeGradient with an InverseCostWeightedUtility of a
        deterministic per-source cost.  Fixing the fantasy rows' source column at the target source is the
        multi-fidelity projection.  The values are differentiable in the quantitative columns of all q + F rows when X
        requires a gradient; a t-batch whose covariance needed jitter raises a NumericalWarning."""
        if cost_by_source is not None and current_value is None:
            raise ValueError("knowledge_gradient: cost_by_source needs current_value")
        if X.dim() < 2:
            raise ValueError("knowledge_gradient expects X of shape [..., q + num_fantasies, d]")
        self.eval()
        nf = int(num_fantasies)
        batch, q_tot, d = X.shape[:-2], int(X.shape[-2]), int(X.shape[-1])
        q = q_tot - nf
        if nf < 1 or q < 1:
            raise ValueError("knowledge_gradient: X has %d rows per t-batch, which does not leave q >= 1 actual rows "
                             "besides num_fantasies = %d >= 1" % (q_tot, nf))
        if q_tot > _engine.MAX_QBATCH:
            raise ValueError("knowledge_gradient: q + num_fantasies = %d exceeds %d" % (q_tot, _engine.MAX_QBATCH))
        if base_samples is None:
            base_samples = sobol_normal_samples(nf, q, seed)
        base = np.ascontiguousarray(torch.as_tensor(base_samples).detach().to("cpu", torch.float64).numpy())
        if base.shape != (nf, q):
            raise ValueError("knowledge_gradient: base_samples must have shape [%d, %d], got %s"
                             % (nf, q, base.shape))
        x = X.reshape(-1, q_tot, d)
        eng, xq, kwargs = self._joint_request(x.detach().double().reshape(-1, d), True)
        kwargs.pop("include_noise")
        kwargs.update(base_samples=base, maximize=bool(maximize))
        if torch.is_grad_enabled() and X.requires_grad:
            v, jitter = _EngineKG.apply(x, eng, xq, q, self._quant_columns(), kwargs)
        else:
            values, _, jitter = eng.kg_qbatch(xq, q, nf, want_grad=False, **kwargs)
            v, jitter = torch.as_tensor(np.asarray(values)), torch.as_tensor(np.asarray(jitter))
        if bool((jitter > 0).any()):
            warnings.warn("A not p.d., added jitter of %.1e to the diagonal" % float(jitter.max()), NumericalWarning)
        dtype = self._out_dtype()
        sgn = 1.0 if maximize else -1.0
        out = sgn * float(self.y_min) + float(self.y_std) * v.to(dtype)
        if current_value is not None:
            out = out - float(current_value)
        if cost_by_source is not None:
            src = x.detach()[:, :q, -1].cpu().double().round().long()
            cost = torch.tensor([[float(cost_by_source[int(s_)]) for s_ in row] for row in src.tolist()],
                                dtype=torch.float64).sum(-1)
            out = out / cost.to(dtype)
        return out.reshape(batch)

    def sample_max_values(self, candidate_set: torch.Tensor, num_samples: int = 10, method: str = "gumbel",
                          maximize: bool = True, seed: int = 0) -> torch.Tensor:
        """``num_samples`` samples [K] of the optimum of f over ``candidate_set`` [M, d] in the original y units: the
        maximum when ``maximize``, else the minimum (botorch's max-value samplers for max-value entropy search; for
        multi-fidelity pass the candidates at the target fidelity).

        ``method="gumbel"`` is botorch's _sample_max_value_Gumbel: the engine finds the quartiles of the maximum under
        the candidates' independent marginals (gpp_max_value_quartiles, the marginals never leave the GPU), a Gumbel
        distribution is fitted to them and sampled at ``num_samples`` uniforms.  ``method="thompson"`` takes the
        optimum over the candidates of each joint posterior draw (``sample_posterior``, M <= MAX_JOINT).  The uniforms
        or normals come from a ``torch.Generator`` seeded with ``seed``."""
        if method not in ("gumbel", "thompson"):
            raise ValueError("sample_max_values: method must be 'gumbel' or 'thompson', got %r" % (method,))
        k = int(num_samples)
        if k < 1:
            raise ValueError("sample_max_values: num_samples must be >= 1, got %d" % k)
        if candidate_set.dim() != 2:
            raise ValueError("sample_max_values expects candidate_set of shape [M, d]")
        gen = torch.Generator().manual_seed(int(seed))
        sgn = 1.0 if maximize else -1.0
        dtype = self._out_dtype()
        with torch.no_grad():
            if method == "thompson":
                if candidate_set.shape[0] > _engine.MAX_JOINT:
                    raise ValueError("sample_max_values: Thompson sampling takes at most %d candidates, got %d"
                                     % (_engine.MAX_JOINT, candidate_set.shape[0]))
                base = torch.randn(k, int(candidate_set.shape[0]), generator=gen, dtype=torch.float64)
                draws = self.sample_posterior(candidate_set, k, base_samples=base)
                return draws.amax(-1) if maximize else draws.amin(-1)
            eng, xq, kwargs = self._joint_request(candidate_set, False)
            y1, y2, y3 = (float(v) for v in np.asarray(eng.max_value_quartiles(
                xq, level_idx=kwargs["level_idx"], mean_idx=kwargs["mean_idx"], maximize=bool(maximize))))
            beta = (y1 - y3) / (math.log(math.log(4.0 / 3.0)) - math.log(math.log(4.0)))
            alpha = y2 + beta * math.log(math.log(2.0))
            u = torch.rand(k, generator=gen, dtype=torch.float64)
            m_sc = alpha - beta * torch.log(-torch.log(u))
            return float(self.y_min) + sgn * float(self.y_std) * m_sc.to(dtype)

    def gibbon(self, X: torch.Tensor, max_values, maximize: bool = True, target_fixed_columns=None, X_pending=None,
               cost_by_source=None) -> torch.Tensor:
        """GIBBON (botorch's qLowerBoundMaxValueEntropy; with ``target_fixed_columns``,
        qMultiFidelityLowerBoundMaxValueEntropy) of every t-batch of X [..., q, d]: values [...] in nats
        (gpp_gibbon_qbatch).  The value is the diversity of the batch (1/2 log det of the correlation matrix of its
        noisy observations) plus, per row, 1/2 log of the variance of its observation over that variance given that
        f at the row (at its target-fidelity copy) stays below the optimum, averaged over ``max_values`` [K] (samples
        of the optimum in the original y units, e.g. from ``sample_max_values``).

        ``target_fixed_columns`` ({column: value}, e.g. the source column at the target fidelity, or a continuous
        fidelity column at its target value) gives the target rows: X with those columns overwritten, so a held
        quantitative column passes no gradient through the target rows.  ``X_pending`` [p, d] is appended to every t-batch and the value
        becomes the gain alpha([X_t, X_pending]) - alpha(X_pending).  ``cost_by_source`` ({source: cost} or a
        sequence indexed by source) then divides that gain by the summed cost of X_t's rows, whose source is the last
        column.  The values are differentiable in the quantitative columns of X when it requires a gradient; a
        t-batch whose covariance needed jitter raises a NumericalWarning."""
        if X.dim() < 2:
            raise ValueError("gibbon expects X of shape [..., q, d]")
        self.eval()
        batch, q, d = X.shape[:-2], int(X.shape[-2]), int(X.shape[-1])
        mv = torch.as_tensor(max_values).detach().to("cpu", torch.float64).reshape(-1)
        if not 1 <= mv.numel() <= _engine.MAX_MC_SAMPLES:
            raise ValueError("gibbon: between 1 and %d max values, got %d" % (_engine.MAX_MC_SAMPLES, mv.numel()))
        sgn = 1.0 if maximize else -1.0
        m_sc = np.ascontiguousarray((sgn * (mv - float(self.y_min)) / float(self.y_std)).numpy())
        pend = None
        if X_pending is not None:
            pend = torch.as_tensor(X_pending).detach().to("cpu", torch.float64).reshape(-1, d)
        q_eff = q + (0 if pend is None else int(pend.shape[0]))
        proj = target_fixed_columns is not None
        if q < 1 or q_eff * (2 if proj else 1) > _engine.MAX_QBATCH:
            raise ValueError("gibbon: %d rows per t-batch (with pending and target rows) is outside [1, %d]"
                             % (q_eff * (2 if proj else 1), _engine.MAX_QBATCH))

        def rows(xa: torch.Tensor) -> torch.Tensor:  # [b, r, d] -> the engine's t-batches [b, r or 2r, d]
            if not proj:
                return xa
            xt = xa.clone()
            for c, v in target_fixed_columns.items():
                xt[:, :, int(c)] = float(v)
            return torch.cat([xa, xt], 1)

        def request(xa: torch.Tensor):
            x_all = rows(xa)
            eng, xq, kwargs = self._joint_request(x_all.reshape(-1, d), True)
            kwargs.pop("include_noise")
            kwargs.update(max_values=m_sc, projected=proj, maximize=bool(maximize))
            return eng, xq, kwargs

        x = X.reshape(-1, q, d)
        xd = x.detach().to("cpu", torch.float64)
        xa = xd if pend is None else torch.cat([xd, pend.expand(xd.shape[0], -1, -1)], 1)
        eng, xq, kwargs = request(xa)
        if torch.is_grad_enabled() and X.requires_grad:
            held = tuple(int(c) for c in target_fixed_columns) if proj else ()
            v, jitter = _EngineGIBBON.apply(x, eng, xq, (q_eff, held), self._quant_columns(), kwargs)
        else:
            values, _, jitter = eng.gibbon_qbatch(xq, q_eff, want_grad=False, **kwargs)
            v, jitter = torch.as_tensor(np.asarray(values)), torch.as_tensor(np.asarray(jitter))
        if pend is not None:
            eng, xq, kwargs = request(pend[None])
            base, _, jit_p = eng.gibbon_qbatch(xq, int(pend.shape[0]), want_grad=False, **kwargs)
            v = v - float(np.asarray(base)[0])
            jitter = torch.cat([jitter, torch.as_tensor(np.asarray(jit_p))])
        if bool((jitter > 0).any()):
            warnings.warn("A not p.d., added jitter of %.1e to the diagonal" % float(jitter.max()), NumericalWarning)
        out = v.to(self._out_dtype())
        if cost_by_source is not None:
            src = xd[:, :, -1].round().long()
            cost = torch.tensor([[float(cost_by_source[int(s_)]) for s_ in row] for row in src.tolist()],
                                dtype=torch.float64).sum(-1)
            out = out / cost.to(out.dtype)
        return out.reshape(batch)

    def reset_parameters(self) -> None:
        """Reset parameters by sampling from the priors (gpregression.py:168-174)."""
        for _, module, prior, closure, setting_closure in self.named_priors():
            if not closure(module).requires_grad:
                continue
            setting_closure(module, prior.expand(closure(module).shape).sample())
