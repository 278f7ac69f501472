"""Host-side building blocks the GP+ model classes are composed from.

The reference composes gpytorch objects (``Module`` with priors and constraints, kernels, means,
likelihoods); gpytorch is not a dependency here.  These classes keep the pieces of that interface
the GP+ hot path relies on -- parameter / prior names and ordering (optim/mll_scipy.py:40-43,
:70-79, :130-138), constraint transforms (models/gpregression.py:59,108-111,
models/gp_plus.py:242-272) -- and are *descriptors*: they own the raw parameters and say which
sm_100a kernel family evaluates them.  No covariance arithmetic happens in Python.
"""
from __future__ import annotations

import math
import warnings
from collections import OrderedDict
from typing import Callable, Iterator, Optional, Tuple

import torch
from torch import nn
from torch.distributions import LogNormal, Normal

from . import _engine


# ----------------------------------------------------------------------------------------------
# errors / settings (gpytorch.utils.errors, gpytorch.settings)
NotPSDError = _engine.NotPSDError
NanError = _engine.NanError


class NumericalWarning(RuntimeWarning):
    """gpytorch.utils.warnings.NumericalWarning: jitter was added to make a covariance positive definite."""


class _Flag:
    """Context manager stand-in for gpytorch.settings.fast_computations: the engine always uses the
    exact Cholesky path, so the flag is accepted and ignored."""

    def __init__(self, *args, **kwargs):
        pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        return False


class settings:  # noqa: N801  (mirrors ``gpytorch.settings``)
    fast_computations = _Flag
    fast_pred_var = _Flag
    cholesky_jitter = _Flag
    min_variance = 1e-10


# ----------------------------------------------------------------------------------------------
# constraints
def _softplus(x):
    return torch.nn.functional.softplus(x)


def _inv_softplus(x):
    return x + torch.log(-torch.expm1(-x))


class Interval(nn.Module):
    def __init__(self, lower_bound, upper_bound, transform=torch.sigmoid, inv_transform=None, initial_value=None):
        super().__init__()
        self.lower_bound = torch.as_tensor(float(lower_bound))
        self.upper_bound = torch.as_tensor(float(upper_bound))
        self._transform = transform
        self._inv_transform = inv_transform
        self.initial_value = initial_value

    @property
    def enforced(self):
        return self._transform is not None

    def transform(self, raw):
        if not self.enforced:
            return raw
        lo, hi = float(self.lower_bound), float(self.upper_bound)
        return self._transform(raw) * (hi - lo) + lo

    def inverse_transform(self, value):
        if not self.enforced:
            return value
        if self._inv_transform is None:
            raise RuntimeError("constraint has no inverse transform")
        lo, hi = float(self.lower_bound), float(self.upper_bound)
        return self._inv_transform((value - lo) / (hi - lo))


class GreaterThan(Interval):
    """value = lower_bound + transform(raw)   (noise constraint, gpregression.py:59)."""

    def __init__(self, lower_bound, transform=_softplus, inv_transform=_inv_softplus, initial_value=None):
        super().__init__(lower_bound, math.inf, transform, inv_transform, initial_value)

    def transform(self, raw):
        if not self.enforced:
            return raw
        return self._transform(raw) + float(self.lower_bound)

    def inverse_transform(self, value):
        if not self.enforced:
            return value
        return self._inv_transform(value - float(self.lower_bound))


class Positive(GreaterThan):
    def __init__(self, transform=_softplus, inv_transform=_inv_softplus, initial_value=None):
        super().__init__(0.0, transform, inv_transform, initial_value)

    def transform(self, raw):
        return self._transform(raw) if self.enforced else raw

    def inverse_transform(self, value):
        return self._inv_transform(value) if self.enforced else value


# ----------------------------------------------------------------------------------------------
# priors
class Prior:
    """Marker base: a torch Distribution usable with ``Module.register_prior``."""

    def transform(self, x):
        return x


def _f64(v):
    """Prior constants are held in float64 so log-densities carry no float32 rounding of log(scale)."""
    return torch.as_tensor(v, dtype=torch.float64) if not torch.is_tensor(v) else v.to(torch.float64)


class NormalPrior(Prior, Normal):
    def __init__(self, loc, scale, validate_args=None):
        Normal.__init__(self, loc=_f64(loc), scale=_f64(scale), validate_args=validate_args)

    def expand(self, batch_shape, _instance=None):
        batch_shape = torch.Size(batch_shape)
        return NormalPrior(self.loc.expand(batch_shape), self.scale.expand(batch_shape))


class LogNormalPrior(Prior, LogNormal):
    def __init__(self, loc, scale, validate_args=None):
        LogNormal.__init__(self, loc=_f64(loc), scale=_f64(scale), validate_args=validate_args)

    def expand(self, batch_shape, _instance=None):
        batch_shape = torch.Size(batch_shape)
        return LogNormalPrior(self.loc.expand(batch_shape), self.scale.expand(batch_shape))


# ----------------------------------------------------------------------------------------------
class Module(nn.Module):
    """nn.Module + named priors + named constraints (the subset of gpytorch.Module GP+ touches)."""

    def __init__(self):
        super().__init__()
        self._priors = OrderedDict()
        self._constraints_by_param = OrderedDict()

    # -- priors --
    def register_prior(self, name: str, prior, param_or_closure, setting_closure: Optional[Callable] = None):
        if isinstance(param_or_closure, str):
            pname = param_or_closure
            if not hasattr(self, pname):
                raise AttributeError("Unknown parameter %r for %s" % (pname, self.__class__.__name__))

            def closure(module, _p=pname):
                return getattr(module, _p)

            if setting_closure is None:
                def setting_closure(module, value, _p=pname):  # noqa: E306
                    return module.initialize(**{_p: value})
        else:
            closure = param_or_closure
        self._priors[name] = (prior, closure, setting_closure)

    def named_priors(self, memo=None, prefix: str = "") -> Iterator[Tuple[str, nn.Module, object, Callable, Callable]]:
        """(name, module, prior, closure, setting_closure): depth-first in module-registration order, the
        module's own priors first -- the same order as ``named_parameters`` (SURVEY A.8)."""
        if memo is None:
            memo = set()
        for mprefix, module in self.named_modules(prefix=prefix):
            for name, (prior, closure, setter) in getattr(module, "_priors", {}).items():
                if prior is None or id(prior) in memo:
                    continue
                memo.add(id(prior))
                yield (mprefix + ("." if mprefix else "") + name, module, prior, closure, setter)

    # -- constraints --
    def register_constraint(self, param_name: str, constraint):
        if param_name not in self._parameters:
            raise RuntimeError("Attempting to register constraint for nonexistent parameter %s" % param_name)
        self._constraints_by_param[param_name] = constraint
        self.add_module(param_name + "_constraint", constraint)

    def constraint_for(self, param_name: str):
        return self._constraints_by_param.get(param_name)

    # -- initialise raw or constrained values by name --
    def initialize(self, **kwargs):
        for name, val in kwargs.items():
            if isinstance(val, (int, float)):
                val = float(val)
            if name in self._parameters:
                p = self._parameters[name]
                v = torch.as_tensor(val, dtype=p.dtype, device=p.device)
                p.data.copy_(v.expand_as(p) if v.numel() == 1 or v.shape != p.shape else v)
            elif hasattr(type(self), name) and isinstance(getattr(type(self), name), property):
                setattr(self, name, val)
            elif "." in name:
                head, rest = name.split(".", 1)
                getattr(self, head).initialize(**{rest: val})
            else:
                raise AttributeError("Unknown parameter %s for %s" % (name, self.__class__.__name__))
        return self


# ----------------------------------------------------------------------------------------------
# kernels (descriptors)
FAMILY_EXPSQ, FAMILY_MATERN32, FAMILY_MATERN52 = _engine.KERNEL_EXPSQ, _engine.KERNEL_MATERN32, _engine.KERNEL_MATERN52


class Kernel(Module):
    has_lengthscale = False
    family = None  # engine kernel family of a stationary leaf kernel

    def __init__(self, ard_num_dims: Optional[int] = None, active_dims=None, lengthscale_prior=None,
                 lengthscale_constraint=None, batch_shape=torch.Size(), **kwargs):
        super().__init__()
        if active_dims is not None and not torch.is_tensor(active_dims):
            active_dims = torch.tensor(active_dims, dtype=torch.long)
        self.register_buffer("active_dims", active_dims)
        self.ard_num_dims = ard_num_dims
        if self.has_lengthscale:
            nd = 1 if ard_num_dims is None else ard_num_dims
            self.register_parameter("raw_lengthscale", nn.Parameter(torch.zeros(*batch_shape, 1, nd)))
            if lengthscale_constraint is None:
                lengthscale_constraint = Positive()
            self.register_constraint("raw_lengthscale", lengthscale_constraint)
            if lengthscale_prior is not None:
                self.register_prior("lengthscale_prior", lengthscale_prior, "lengthscale")

    @property
    def lengthscale(self):
        if not self.has_lengthscale:
            return None
        return self.raw_lengthscale_constraint.transform(self.raw_lengthscale)

    @lengthscale.setter
    def lengthscale(self, value):
        value = torch.as_tensor(value, dtype=self.raw_lengthscale.dtype)
        raw = self.raw_lengthscale_constraint.inverse_transform(value)
        self.raw_lengthscale.data.copy_(raw.expand_as(self.raw_lengthscale))

    def distance_weights(self) -> torch.Tensor:
        """w_d such that the family function is applied to s = sum_d w_d dx_d^2 (differentiable in raw)."""
        raise NotImplementedError

    def __mul__(self, other):
        parts = []
        for k in (self, other):
            parts.extend(list(k.kernels) if isinstance(k, ProductKernel) else [k])
        return ProductKernel(*parts)

    def leaf_kernels(self):
        return [self]

    def forward(self, x1, x2=None, **params):
        from ._dense import dense_kernel  # engine-backed dense evaluation
        return dense_kernel(self, x1, x2)

    def __call__(self, x1, x2=None, **params):
        return _LazyKernel(self, x1, x2)


class _LazyKernel:
    """``covar_module(x)`` result: dense evaluation happens on the GPU when ``evaluate()`` is called."""

    def __init__(self, kernel, x1, x2):
        self.kernel, self.x1, self.x2 = kernel, x1, x2
        self._dtype = None

    def to(self, *args, **kwargs):
        for a in list(args) + list(kwargs.values()):
            if isinstance(a, torch.dtype):
                self._dtype = a
        return self

    def evaluate(self):
        k = self.kernel.forward(self.x1, self.x2)
        return k if self._dtype is None else k.to(self._dtype)

    to_dense = evaluate


class RBFKernel(Kernel):
    """k = exp(-1/2 sum (dx/l)^2)."""
    has_lengthscale = True
    family = FAMILY_EXPSQ

    def distance_weights(self):
        ls = self.lengthscale.reshape(-1)
        return 0.5 / (ls * ls)


class MaternKernel(Kernel):
    has_lengthscale = True

    def __init__(self, nu: float = 2.5, **kwargs):
        if nu not in (1.5, 2.5):
            raise RuntimeError("nu expected to be 1.5 or 2.5 (the engine has no Matern-1/2 family)")
        super().__init__(**kwargs)
        self.nu = nu

    @property
    def family(self):
        return FAMILY_MATERN32 if self.nu == 1.5 else FAMILY_MATERN52

    def distance_weights(self):
        ls = self.lengthscale.reshape(-1)
        return 1.0 / (ls * ls)


class ProductKernel(Kernel):
    def __init__(self, *kernels):
        super().__init__()
        self.kernels = nn.ModuleList(kernels)

    def leaf_kernels(self):
        out = []
        for k in self.kernels:
            out.extend(k.leaf_kernels())
        return out


class ScaleKernel(Kernel):
    """K = outputscale * base_kernel   (gpregression.py:108-111)."""

    def __init__(self, base_kernel, outputscale_prior=None, outputscale_constraint=None, **kwargs):
        super().__init__(**kwargs)
        self.base_kernel = base_kernel
        self.register_parameter("raw_outputscale", nn.Parameter(torch.zeros(())))
        if outputscale_constraint is None:
            outputscale_constraint = Positive()
        self.register_constraint("raw_outputscale", outputscale_constraint)
        if outputscale_prior is not None:
            self.register_prior("outputscale_prior", outputscale_prior, "outputscale")

    @property
    def outputscale(self):
        return self.raw_outputscale_constraint.transform(self.raw_outputscale)

    @outputscale.setter
    def outputscale(self, value):
        value = torch.as_tensor(value, dtype=self.raw_outputscale.dtype)
        self.raw_outputscale.data.copy_(self.raw_outputscale_constraint.inverse_transform(value))

    def leaf_kernels(self):
        return self.base_kernel.leaf_kernels()


# ----------------------------------------------------------------------------------------------
# means
class Mean(Module):
    pass


class ZeroMean(Mean):
    def forward(self, x):
        return torch.zeros(x.shape[:-1], dtype=x.dtype, device=x.device)


class ConstantMean(Mean):
    def __init__(self, prior=None, batch_shape=torch.Size()):
        super().__init__()
        self.register_parameter("constant", nn.Parameter(torch.zeros(*batch_shape, 1)))
        if prior is not None:
            self.register_prior("mean_prior", prior, "constant")

    def forward(self, x):
        return self.constant.expand(x.shape[:-1])


# ----------------------------------------------------------------------------------------------
# likelihoods
class HomoskedasticNoise(Module):
    def __init__(self, noise_prior=None, noise_constraint=None, batch_shape=torch.Size(), num_tasks: int = 1):
        super().__init__()
        if noise_constraint is None:
            noise_constraint = GreaterThan(1e-4)
        self.register_parameter("raw_noise", nn.Parameter(torch.zeros(*batch_shape, num_tasks)))
        self.register_constraint("raw_noise", noise_constraint)
        if noise_prior is not None:
            self.register_prior("noise_prior", noise_prior, "noise")

    @property
    def noise(self):
        return self.raw_noise_constraint.transform(self.raw_noise)

    @noise.setter
    def noise(self, value):
        value = torch.as_tensor(value, dtype=self.raw_noise.dtype)
        raw = self.raw_noise_constraint.inverse_transform(value)
        self.raw_noise.data.copy_(raw.expand_as(self.raw_noise))


class _GaussianLikelihoodBase(Module):
    def __init__(self, noise_covar):
        super().__init__()
        self.noise_covar = noise_covar

    @property
    def noise(self):
        return self.noise_covar.noise

    @noise.setter
    def noise(self, value):
        self.noise_covar.initialize(noise=value)

    @property
    def raw_noise(self):
        return self.noise_covar.raw_noise

    @raw_noise.setter
    def raw_noise(self, value):
        self.noise_covar.initialize(raw_noise=value)


class GaussianLikelihood(_GaussianLikelihoodBase):
    def __init__(self, noise_prior=None, noise_constraint=None, batch_shape=torch.Size(), **kwargs):
        super().__init__(HomoskedasticNoise(noise_prior, noise_constraint, batch_shape, 1))


# ----------------------------------------------------------------------------------------------
class MultivariateNormal:
    """Mean vector + dense covariance, the two things GP+ callers read back."""

    def __init__(self, mean, covariance_matrix):
        self.mean = mean
        self.loc = mean
        self._covar = covariance_matrix

    @property
    def covariance_matrix(self):
        return self._covar

    @property
    def lazy_covariance_matrix(self):
        return self._covar

    @property
    def variance(self):
        return torch.diagonal(self._covar, dim1=-2, dim2=-1).clamp_min(settings.min_variance)

    @property
    def stddev(self):
        return self.variance.sqrt()

    def rsample(self, sample_shape=torch.Size(), base_samples=None):
        """Draws [*sample_shape, *batch, q]: mean + L e with L the Cholesky factor of each q x q covariance block
        (gpytorch's MultivariateNormal.rsample).  ``base_samples`` e defaults to standard normal draws; a block that is
        not positive definite gets the psd_safe_cholesky jitter (1e-8, 1e-7, 1e-6) and a NumericalWarning, the other
        blocks none."""
        shape = torch.Size(sample_shape) + self.mean.shape
        if base_samples is None:
            base_samples = torch.randn(shape, dtype=self.mean.dtype, device=self.mean.device)
        elif tuple(base_samples.shape) != tuple(shape):
            raise ValueError("base_samples must have shape %s, got %s" % (tuple(shape), tuple(base_samples.shape)))
        L = _psd_safe_cholesky(self._covar)
        return self.mean + (L @ base_samples.to(self.mean.dtype).unsqueeze(-1)).squeeze(-1)


def _psd_safe_cholesky(A):
    """Batched Cholesky factor; blocks that fail get the smallest jitter of the ladder that lets them factor."""
    L, info = torch.linalg.cholesky_ex(A)
    bad = info != 0
    if not bool(bad.any()):
        return L
    eye = torch.eye(A.shape[-1], dtype=A.dtype, device=A.device)
    for jitter in (1e-8, 1e-7, 1e-6):
        Lj, info_j = torch.linalg.cholesky_ex(A + jitter * eye)
        fix = bad & (info_j == 0)
        if bool(fix.any()):
            warnings.warn("A not p.d., added jitter of %.1e to the diagonal" % jitter, NumericalWarning)
            L = torch.where(fix[..., None, None], Lj, L)
            bad = bad & ~fix
        if not bool(bad.any()):
            return L
    raise NotPSDError("Matrix not positive definite after repeatedly adding jitter up to 1.0e-06.")
