"""``GP_Plus``: mixed-variable / multi-fidelity GP with a learned latent map for categorical inputs.

Mirrors the hot-path surface of models/gp_plus.py of the reference: constructor arguments and
validation (:79-182), index bookkeeping (:184-215), the kernel tree -- fixed-lengthscale RBF on the
latent coordinates times an ARD kernel on the quantitative columns (:219-303) --, the one-hot /
level-combination table (:1027-1073), the latent map ``FFNN`` / ``Linear_MAP`` whose weights are
registered on the model as ``latent[...]`` with N(0,1) priors (:1227-1265, :1456-1461), the constant /
zero / multiple-constant mean functions (:488-544), ``fit`` (:547-599) and ``predict`` (:621-628).

Differences by design: there is no per-row Python work per evaluation (the level-combination index
of every training row is computed once), and no dense matrix is ever built in Python -- the model
hands natural hyper-parameters to ``libgpplus_b200.so``.  Research variants that are outside the
accelerated path (probabilistic embedding, calibration, NN / polynomial means, several separate
latent maps) raise ``NotImplementedError`` instead of silently running something else.
"""
from __future__ import annotations

import math
import warnings
from typing import Dict, List, Optional

import numpy as np
import torch
import torch.nn.functional as F
from torch import nn

from .. import kernels
from .._compat import ConstantMean, Module as _CompatModule, MultivariateNormal, NormalPrior, Positive, ZeroMean
from ..optim import fit_model_continuation, fit_model_scipy, fit_model_torch
from ..preprocessing import setlevels
from ..priors import MollifiedUniformPrior
from ..utils import data_type_check
from .gpregression import GPR

_QUANT_CLASSES = ("Rough_RBF", "RBFKernel", "Matern32Kernel", "Matern12Kernel", "Matern52Kernel")


def _rough_ls(x):
    return 2.0 ** (-0.5) * torch.pow(10, -x / 2)


def _rough_ls_inv(x):
    return -2.0 * torch.log10(x / 2.0)


class GP_Plus(GPR):
    """See the reference docstring (models/gp_plus.py:45-78) for the meaning of every argument."""

    # eval-mode behaviour of the reference kept by default: gpytorch's ExactGP.__call__ hands forward() the
    # concatenation [train_inputs, Xtest], and transform_categorical re-ranks its categorical columns with
    # ``setlevels`` (models/gp_plus.py:1081-1082).  Prediction categories are therefore ranked against the sorted
    # unique values of train U test per column -- the identity whenever training holds every level 0..L-1.
    relevel_on_predict = True

    def __init__(
        self,
        train_x: torch.Tensor,
        train_y: torch.Tensor,
        dtype=torch.float,
        device="cpu",
        qual_dict={},
        multiple_noise=False,
        lb_noise: float = 1e-8,
        fix_noise: bool = False,
        fix_noise_val: float = 1e-5,
        quant_correlation_class: str = "Rough_RBF",
        fixed_length_scale: bool = False,
        fixed_length_scale_val=torch.tensor([1.0]),
        encoding_type="one-hot",
        embedding_dim: int = 2,
        separate_embedding=[],
        embedding_type="deterministic",
        NN_layers_embedding: list = [],
        m_gp="single_constant",
        m_gp_ref="zero",
        NN_layers_m_gp=[],
        calibration_type="deterministic",
        calibration_id=[],
        mean_prior_cal=None,
        std_prior_cal=None,
        interval_score=False,
        num_pass_train=1,
        num_pass_pred=1,
        seed_number=1,
    ) -> None:
        self.interval_score = interval_score
        self.tkwargs = {"dtype": dtype, "device": torch.device(device)}
        self.mean_prior_cal = [0 for _ in calibration_id] if mean_prior_cal is None else mean_prior_cal
        self.std_prior_cal = [1 for _ in calibration_id] if std_prior_cal is None else std_prior_cal
        self.fixed_length_scale_val = fixed_length_scale_val.to(dtype=dtype) if fixed_length_scale else None

        train_x = data_type_check(train_x)
        train_y = data_type_check(train_y)
        if not isinstance(qual_dict, dict):
            raise ValueError("qual_dict should be a dictionary.")
        if multiple_noise not in [True, False]:
            raise ValueError("multiple_noise should be either True or False.")
        if not isinstance(embedding_dim, int):
            raise ValueError("embedding_dim should be an integer.")
        if quant_correlation_class not in _QUANT_CLASSES:
            raise ValueError("quant_correlation_class should be 'Rough_RBF', 'RBFKernel', 'Matern32Kernel', "
                             "'Matern12Kernel','Matern52Kernel'.")
        if fix_noise not in [True, False]:
            raise ValueError("fix_noise should be either True or False.")
        if not isinstance(NN_layers_embedding, list) or not all(isinstance(i, int) for i in NN_layers_embedding):
            raise ValueError("NN_layers_embedding should be a list of integers representing the number of neurons "
                             "in each layer.")
        if encoding_type != "one-hot":
            raise ValueError("encoding_type should be 'one-hot'.")
        if embedding_type not in ["deterministic", "probabilistic"]:
            raise ValueError("embedding_type should be either 'deterministic' or 'probabilistic'.")
        if not isinstance(separate_embedding, list) or not all(isinstance(i, int) for i in separate_embedding):
            raise ValueError("separate_embedding should be a list with integers showing the number of categorical "
                             "inputs to be considered in a separate manifold in each layer.")
        if not isinstance(NN_layers_m_gp, list) or not all(isinstance(i, int) for i in NN_layers_m_gp):
            raise ValueError("NN_layers_m_gp should be a list with integers representing the number of neurons in "
                             "each layer for the mean function.")
        if not isinstance(calibration_id, list) or not all(isinstance(i, int) for i in calibration_id):
            raise ValueError("calibration_id should be a list where each entry shows the column number in the "
                             "dataset that the calibration parameters are assigned to.")
        # variants outside the accelerated hot path (SURVEY section 2, row 1)
        if calibration_type == "probabilistic" or len(calibration_id) > 0:
            raise NotImplementedError("calibration parameters are outside the B200 engine's scope")
        if len(separate_embedding) > 0:
            raise NotImplementedError("separate_embedding: the reference only feeds the last latent map into the "
                                      "kernel (models/gp_plus.py:410-437); use the default shared map")
        if quant_correlation_class == "Matern12Kernel":
            raise RuntimeError("Matern12Kernel not an allowed kernel")  # as models/gp_plus.py:236-241

        train_x = self.fill_nan_with_mean(train_x, calibration_id)
        self.seed = seed_number
        self.calibration_id = calibration_id
        self.calibration_type = calibration_type
        qual_dict_list = list(qual_dict.keys())
        quant_index = sorted(set(range(train_x.shape[-1])).difference(qual_dict_list))
        num_levels_per_var = list(qual_dict.values())
        lm_columns = list(set(qual_dict_list).difference(separate_embedding))
        qual_kernel_columns = [*separate_embedding, lm_columns] if len(lm_columns) > 0 else separate_embedding
        train_y = train_y.reshape(-1)
        noise_indices = list(range(0, num_levels_per_var[-1])) if multiple_noise else []

        if len(qual_dict_list) == 1 and num_levels_per_var[0] < 2:
            quant_index = quant_index + [qual_dict_list[0]]
            qual_dict_list = []
            embedding_dim = 0
        if len(qual_dict_list) == 0:
            embedding_dim = 0
            qual_kernel_columns = []

        qual_kernels = []
        if len(qual_dict_list) > 0:
            for i in range(len(qual_kernel_columns)):
                qk = kernels.RBFKernel(active_dims=torch.arange(embedding_dim) + embedding_dim * i)
                qk.initialize(lengthscale=1.0)
                qk.raw_lengthscale.requires_grad_(False)
                qual_kernels.append(qk)

        quant_kernel = None
        if len(quant_index) == 0:
            correlation_kernel = qual_kernels[0]
            for extra in qual_kernels[1:]:
                correlation_kernel = correlation_kernel * extra
        else:
            dims = len(qual_kernel_columns) * embedding_dim + torch.arange(len(quant_index))
            if quant_correlation_class == "RBFKernel":
                quant_kernel = kernels.RBFKernel(
                    ard_num_dims=len(quant_index), active_dims=dims,
                    lengthscale_constraint=Positive(transform=torch.exp, inv_transform=torch.log))
                quant_kernel.register_prior(
                    "lengthscale_prior", MollifiedUniformPrior(math.log(0.1), math.log(10)), "raw_lengthscale")
            else:
                # 'Rough_RBF' is an RBFKernel with l = 2^-1/2 10^(-omega/2), i.e. exp(-sum 10^omega dx^2)
                cls = {"Rough_RBF": kernels.RBFKernel, "Matern32Kernel": kernels.Matern32Kernel,
                       "Matern52Kernel": kernels.Matern52Kernel}[quant_correlation_class]
                quant_kernel = cls(ard_num_dims=len(quant_index), active_dims=dims,
                                   lengthscale_constraint=Positive(transform=_rough_ls, inv_transform=_rough_ls_inv))
                quant_kernel.register_prior("lengthscale_prior", NormalPrior(-3.0, 3.0), "raw_lengthscale")
            if len(qual_dict_list) > 0:
                temp = qual_kernels[0]
                for extra in qual_kernels[1:]:
                    temp = temp * extra
                correlation_kernel = temp * quant_kernel
            else:
                correlation_kernel = quant_kernel

        super().__init__(train_x=train_x, train_y=train_y, noise_indices=noise_indices,
                         correlation_kernel=correlation_kernel, fix_noise=fix_noise, fix_noise_val=fix_noise_val,
                         lb_noise=lb_noise)
        # shortcuts into the kernel tree; object.__setattr__ keeps them out of the module registry so that
        # named_parameters / state_dict keep the reference's names (covar_module.base_kernel.kernels.1...)
        object.__setattr__(self, "_quant_cols", list(quant_index))
        object.__setattr__(self, "_qual_cols", list(qual_dict_list))
        object.__setattr__(self, "_quant", quant_kernel)
        object.__setattr__(self, "_latent_kernel", qual_kernels[0] if qual_kernels else None)
        self._quant_class_name = quant_correlation_class

        self.register_buffer("quant_index", torch.tensor(quant_index, dtype=torch.long))
        self.register_buffer("qual_dict_list", torch.tensor(qual_dict_list, dtype=torch.long))
        self.qual_kernel_columns = qual_kernel_columns
        self.num_levels_per_var = num_levels_per_var
        self.embedding_dim = embedding_dim
        self.encoding_type = encoding_type
        self.embedding_type = embedding_type
        self.perm, self.zeta, self.perm_dict, self.A_matrix = [], [], [], []
        self.count = train_x.size()[0]
        self.num_pass_train, self.num_pass_pred = num_pass_train, num_pass_pred
        self._level_strides = None
        if len(qual_kernel_columns) > 0:
            cols = qual_kernel_columns[-1]
            cat = [num_levels_per_var[qual_dict_list.index(k)] for k in cols]
            zeta, perm, perm_dict = self.zeta_matrix(num_levels=cat, embedding_dim=embedding_dim)
            self.zeta.append(zeta)
            self.perm.append(perm)
            self.perm_dict.append(perm_dict)
            if embedding_type == "probabilistic":
                # variational encoder: each level combination gets a 2-D Gaussian N(mu, L L^T) in the latent space,
                # sampled once per forward pass with a seeded epsilon (gp_plus.py:347-349, 414-437, 1373-1413);
                # registered as the sub-module ``A_matrix`` so its weights pack after the kernel parameters
                if embedding_dim != 2:
                    raise ValueError("the probabilistic embedding is two-dimensional (gp_plus.py:1387-1412)")
                self.A_matrix = Variational_Encoder(input_size=sum(cat), num_classes=5, layers=NN_layers_embedding
                                                    ).to(dtype=dtype)
                object.__setattr__(self, "_latent_map", None)
            else:
                latent_map = FFNN(self, input_size=sum(cat), num_classes=embedding_dim, layers=NN_layers_embedding,
                                  name="latent" + str(cols)).to(dtype=dtype)
                self.A_matrix.append(latent_map)
                object.__setattr__(self, "_latent_map", latent_map)
            strides = np.ones(len(cat), dtype=np.int64)
            for k in range(len(cat) - 2, -1, -1):
                strides[k] = strides[k + 1] * cat[k + 1]
            self._level_strides = (np.asarray(cat, dtype=np.int64), strides)

        if fixed_length_scale:
            self.covar_module.base_kernel.raw_lengthscale.data = self.fixed_length_scale_val
            self.covar_module.base_kernel.raw_lengthscale.requires_grad = False

        self.m_gp = m_gp
        self.m_gp_ref = m_gp_ref
        self.num_sources = int(torch.max(train_x[:, -1]))
        if m_gp in ("single_constant", "single_zero"):
            self.single_m_gp_register(train_x.shape[1], m_gp_type=m_gp, wm="mean_module")
        elif m_gp == "multiple_constant":
            if m_gp_ref not in ("zero", "constant"):
                raise NotImplementedError("m_gp_ref must be 'zero' or 'constant' for the device mean gather")
            for i in range(self.num_sources + 1):
                kind = "single_" + m_gp_ref if i == 0 else "single_constant"
                self.single_m_gp_register(train_x.shape[1], m_gp_type=kind, wm="mean_module_" + str(i))
        elif m_gp.startswith("single") or m_gp.startswith("multi") or m_gp == "neural_network":
            raise NotImplementedError("mean function %r is outside the B200 engine's scope (constant, zero and "
                                      "multiple_constant are supported)" % m_gp)
        else:
            raise ValueError('The "m_gp" argument must start with "multi", "single", or "neural_network".')
        for prm in self.parameters():  # parameters follow ``dtype``; data buffers keep the dtype of train_y
            prm.data = prm.data.to(dtype)

    # ------------------------------------------------------------------------------------------
    # engine plumbing overrides
    def _quant_columns(self) -> List[int]:
        return self._quant_cols

    def _quant_kernel(self):
        return self._quant

    def _level_index(self, x: torch.Tensor, training: bool, relevel_labels=None) -> Optional[np.ndarray]:
        """Row of the level-combination table per point (perm_dict lookup, gp_plus.py:1085) -- vectorised
        mixed-radix index, identical to the itertools.product order of ``zeta_matrix``.

        In eval mode the reference ranks the categorical columns of ``[train_inputs, x]`` (see
        ``relevel_on_predict``); ``relevel_labels`` (one array of values per categorical column) replaces the
        values of ``x`` in that union: callers that score a chunk of a larger batch pass the labels of the whole
        batch so that the chunk is ranked exactly as the reference would rank the batch."""
        if self._level_strides is None:
            return None
        cols = self.qual_kernel_columns[-1]
        cat = x[:, cols].detach().cpu().type(torch.int64).numpy()
        if not training and self.relevel_on_predict:
            train_labels = self._train_labels()
            c = np.empty_like(cat)
            for k in range(len(cols)):
                seen = cat[:, k] if relevel_labels is None else np.asarray(relevel_labels[k], dtype=np.int64)
                union = np.union1d(train_labels[k], seen)
                c[:, k] = np.searchsorted(union, cat[:, k])
        else:
            c = cat
        levels, strides = self._level_strides
        if (c < 0).any() or (c >= levels[None, :]).any():
            raise ValueError("The categorical input (or source indices) are not defined properly. They should be "
                             "integer values starting from zero. To solve the issue, you can use the 'setlevels' "
                             "function, which is a preprocessing function.")
        return (c * strides[None, :]).sum(1).astype(np.int32)

    def _train_labels(self):
        """Sorted unique values (int64) of every categorical column of the training inputs."""
        cached = self.__dict__.get("_train_labels_cache")
        if cached is None:
            cols = self.qual_kernel_columns[-1]
            cat = self.train_inputs[0][:, cols].detach().cpu().type(torch.int64).numpy()
            cached = [np.unique(cat[:, k]) for k in range(len(cols))]
            self.__dict__["_train_labels_cache"] = cached
        return cached

    def _relevel_labels(self, x: torch.Tensor):
        """Unique values of every categorical column of ``x`` truncated to int64 (the part of the eval-mode
        ``setlevels`` ranking contributed by ``x``), or None when the model has no categorical input."""
        if self._level_strides is None:
            return None
        cols = self.qual_kernel_columns[-1]
        cat = x[:, cols].detach().cpu().type(torch.int64).numpy()
        return [np.unique(cat[:, k]) for k in range(len(cols))]

    def _latent_table(self) -> Optional[torch.Tensor]:
        if self._level_strides is None:
            return None
        dtype = self.covar_module.raw_outputscale.dtype
        if self.embedding_type == "probabilistic":
            return self._sampled_latent_tables(dtype) / self._latent_kernel.lengthscale.reshape(-1)[0]
        z = self._latent_map(self.zeta[-1].to(dtype))
        return z / self._latent_kernel.lengthscale.reshape(-1)[0]

    def _latent_passes(self) -> int:
        """Latent tables averaged into the covariance: ``num_pass_train`` forward passes in training mode,
        ``num_pass_pred`` in eval mode (gp_plus.py:387-393); 1 for the deterministic map."""
        if self.embedding_type != "probabilistic" or self._level_strides is None:
            return 1
        return max(1, int(self.num_pass_train if self.training else self.num_pass_pred))

    def _sampled_latent_tables(self, dtype) -> torch.Tensor:
        """[passes, n_combo, 2] latent positions of the probabilistic embedding, one table per forward pass.

        Mirrors gp_plus.py:388-437: the generator is re-seeded with ``seed_number`` at every forward, each pass
        draws ``epsilon ~ N(0, 1)`` of shape [u, 2] for the u level combinations PRESENT in the training inputs
        (``torch.unique(one_hot_rows, dim=0)`` order), the encoder turns (one-hot row, epsilon) into a position, and
        the positions are written into a float32 buffer (``x_raw = torch.zeros(n, 2)``) before they reach the kernel,
        i.e. rounded to float32 -- kept, with a straight-through gradient.  A private generator is used instead of
        re-seeding torch's global one."""
        present = self.__dict__.get("_present_combos")
        if present is None:
            lv = self._level_index(self.train_inputs[0], True)
            rows = self.zeta[-1][np.unique(lv)]
            uniq = torch.unique(rows, dim=0)  # lexicographic order of the one-hot rows, as the reference gets it
            # combination index of every unique one-hot row
            table = {tuple(r.tolist()): i for i, r in enumerate(self.zeta[-1])}
            present = (uniq, torch.as_tensor([table[tuple(r.tolist())] for r in uniq], dtype=torch.long))
            self.__dict__["_present_combos"] = present
        uniq, combo = present
        gen = torch.Generator().manual_seed(int(self.seed))
        passes = self._latent_passes()
        n_combo = self.zeta[-1].shape[0]
        tables = []
        for _ in range(passes):
            eps = torch.normal(mean=0.0, std=1.0, size=[uniq.shape[0], 2], generator=gen)
            pos = self.A_matrix(uniq.to(dtype), eps)
            pos = pos + (pos.float().to(pos.dtype) - pos).detach()  # float32 rounding, gradient passes through
            tables.append(torch.zeros(n_combo, 2, dtype=pos.dtype).index_copy(0, combo, pos))
        return torch.stack(tables)

    def _check_combos_seen(self, levels: np.ndarray):
        if self.embedding_type == "probabilistic":
            seen = set(self.__dict__["_present_combos"][1].tolist()) if "_present_combos" in self.__dict__ else None
            if seen is None:
                self._sampled_latent_tables(self.covar_module.raw_outputscale.dtype)
                seen = set(self.__dict__["_present_combos"][1].tolist())
            if not set(np.unique(levels).tolist()) <= seen:
                raise ValueError("probabilistic embedding: a level combination of the prediction inputs does not occur "
                                 "in the training data (the reference samples latent positions for training "
                                 "combinations only, gp_plus.py:419-434)")

    def _mean_layout(self):
        if self.m_gp == "multiple_constant":
            consts = []
            for i in range(self.num_sources + 1):
                mm = getattr(self, "mean_module_" + str(i))
                if isinstance(mm, ConstantMean):
                    consts.append(mm.constant)
            return len(consts), consts
        return super()._mean_layout()

    def _mean_index(self, x: torch.Tensor) -> Optional[np.ndarray]:
        if self.m_gp != "multiple_constant":
            return None
        src = x[:, -1].cpu().numpy().astype(np.int64)
        if (src < 0).any() or (src > self.num_sources).any():
            raise ValueError("source index outside the sources seen in training")
        shift = 1 if isinstance(getattr(self, "mean_module_0"), ZeroMean) else 0
        return (src - shift).astype(np.int32)  # -1 selects the zero mean of the reference source

    # ------------------------------------------------------------------------------------------
    def forward(self, x: torch.Tensor) -> MultivariateNormal:
        """Prior mean and dense covariance at x in float64 (gp_plus.py:386-484); off the hot path."""
        from .._dense import dense_model_covariance
        xc = x.detach().cpu()
        mean_x = self._mean_vector(xc)
        return MultivariateNormal(mean_x, dense_model_covariance(self, xc))

    def _mean_vector(self, x):
        with torch.no_grad():
            n_mean, consts = self._mean_layout()
            out = torch.zeros(x.shape[0], dtype=torch.float64)
            if n_mean == 0:
                return out
            beta = torch.cat([c.reshape(-1) for c in consts]).double()
            idx = self._mean_index(x)
            if idx is None:
                return out + beta[0]
            idx = torch.as_tensor(idx, dtype=torch.long)
            return torch.where(idx >= 0, beta[idx.clamp_min(0)], out)

    def single_m_gp_register(self, size=1, m_gp_type="single_zero", wm="mean_module"):
        if m_gp_type == "single_constant":
            setattr(self, wm, ConstantMean(prior=NormalPrior(0.0, 1)))
        elif m_gp_type == "single_zero":
            setattr(self, wm, ZeroMean())
        else:
            raise NotImplementedError("mean function %r is outside the B200 engine's scope" % m_gp_type)

    # ------------------------------------------------------------------------------------------
    def fit(self, add_prior: bool = True, num_restarts: int = 64, theta0_list: Optional[List[np.ndarray]] = None,
            jac: bool = True, options: Dict = {}, n_jobs: int = -1, method="L-BFGS-B", constraint=False, bounds=False,
            regularization_parameter: List[int] = [0, 0], optim_type="scipy"):
        print("## Learning the model's parameters has started ##")
        if self.tkwargs["device"].type == "cuda" and optim_type != "adam_torch":
            # the reference cannot run its scipy path on CUDA tensors and falls back to Adam
            # (models/gp_plus.py:551-567); here the hyper-parameters always live on the host and every
            # optimiser drives the same GPU engine, so the requested optimiser is honoured.
            warnings.warn("device='cuda': hyper-parameters stay on the host; the GPU engine serves optim_type=%r"
                          % optim_type)
        if optim_type == "scipy":
            fit_model_scipy(self, add_prior, num_restarts, theta0_list, jac, options, n_jobs, method, constraint,
                            bounds, regularization_parameter)
        elif optim_type == "continuation":
            fit_model_continuation(model=self, add_prior=add_prior, num_restarts=num_restarts, criterion="NLL",
                                   initial_noise_var=1, red_factor=math.sqrt(10), options=options, n_jobs=n_jobs,
                                   accuracy=1e-2, method=method, constraint=constraint,
                                   regularization_parameter=regularization_parameter, bounds=bounds)
        elif optim_type == "adam_torch":
            fit_model_torch(model=self, model_param_groups=None, lr_default=0.01, num_iter=100,
                            num_restarts=num_restarts, break_steps=50)
        else:
            raise ValueError(
                'Invalid optim_type. You must choose one of the following: "scipy" (default), "continuation", or '
                '"adam_torch".')
        print("## Learning the model's parameters is successfully finished ##")

    def fill_nan_with_mean(self, train_x, cal_ID):
        if torch.isnan(train_x).any():
            print("There are NaN values in the data, which will be filled with column-wise mean values."
                  if len(cal_ID) == 0 else
                  "There are NaN values in the data, which will be estimated in calibration process")
            col_means = torch.nanmean(train_x, dim=0)
            nan_idx = torch.isnan(train_x)
            train_x[nan_idx] = col_means.repeat(train_x.shape[0], 1)[nan_idx]
        return train_x

    def predict(self, Xtest, return_std=True, include_noise=True):
        Xtest = data_type_check(Xtest)
        with torch.no_grad():
            return super().predict(Xtest, return_std=return_std, include_noise=include_noise)

    def predict_with_grad(self, Xtest, return_std=True, include_noise=True):
        """Reference: ``predict`` without ``torch.no_grad()`` (gp_plus.py:626-628).  When ``Xtest`` requires a gradient
        the mean and std carry an autograd graph back to ``Xtest`` only: the derivatives w.r.t. its quantitative
        columns come from the engine (gpp_predict_grad), its categorical and source columns get zero, and the graph
        does not reach the model's parameters.  First derivatives only.  The values equal ``predict``'s."""
        Xtest = data_type_check(Xtest)
        return super().predict(Xtest, return_std=return_std, include_noise=include_noise)

    def predict_joint(self, Xtest, include_noise=False):
        """Posterior mean [M] and full covariance [M, M] at ``Xtest`` in the original y units (GPR.predict_joint)."""
        Xtest = data_type_check(Xtest)
        with torch.no_grad():
            return super().predict_joint(Xtest, include_noise=include_noise)

    def sample_posterior(self, Xtest, num_samples=1, include_noise=False, base_samples=None, generator=None):
        """``num_samples`` joint posterior draws [S, M] at ``Xtest`` in the original y units (GPR.sample_posterior)."""
        Xtest = data_type_check(Xtest)
        with torch.no_grad():
            return super().sample_posterior(Xtest, num_samples=num_samples, include_noise=include_noise,
                                            base_samples=base_samples, generator=generator)

    def acquisition_qbatch(self, X, kind="qEI", best_f=None, X_baseline=None, beta=None, num_samples=512,
                           base_samples=None, seed=0, maximize=True, observation_noise=False, mc_points=None):
        """Batch acquisition values of the t-batches of ``X`` [..., q, d] in the original y units
        (GPR.acquisition_qbatch: Monte-Carlo qEI / qNEI / qUCB, or qNIPV over ``mc_points``); differentiable in ``X``
        when it requires a gradient, as ``predict_with_grad``."""
        X = data_type_check(X)
        if mc_points is not None:
            mc_points = data_type_check(mc_points)
        return super().acquisition_qbatch(X, kind=kind, best_f=best_f, X_baseline=X_baseline, beta=beta,
                                          num_samples=num_samples, base_samples=base_samples, seed=seed,
                                          maximize=maximize, observation_noise=observation_noise,
                                          mc_points=mc_points)

    def knowledge_gradient(self, X, num_fantasies, base_samples=None, seed=0, maximize=True, current_value=None,
                           cost_by_source=None):
        """One-shot knowledge gradient of the t-batches of ``X`` [..., q + num_fantasies, d] in the original y units,
        optionally net of ``current_value`` and per unit cost of the actual rows' sources (GPR.knowledge_gradient);
        differentiable in ``X`` when it requires a gradient, as ``predict_with_grad``."""
        X = data_type_check(X)
        return super().knowledge_gradient(X, num_fantasies, base_samples=base_samples, seed=seed, maximize=maximize,
                                          current_value=current_value, cost_by_source=cost_by_source)

    def gibbon(self, X, max_values, maximize=True, target_fixed_columns=None, X_pending=None, cost_by_source=None):
        """GIBBON values of the t-batches of ``X`` [..., q, d] in nats, optionally against the target rows of
        ``target_fixed_columns``, net of ``X_pending`` and per unit cost of the rows' sources (GPR.gibbon);
        differentiable in ``X`` when it requires a gradient, as ``predict_with_grad``."""
        X = data_type_check(X)
        return super().gibbon(X, max_values, maximize=maximize, target_fixed_columns=target_fixed_columns,
                              X_pending=X_pending, cost_by_source=cost_by_source)

    def sample_max_values(self, candidate_set, num_samples=10, method="gumbel", maximize=True, seed=0):
        """Samples of the optimum of f over ``candidate_set`` [M, d] in the original y units (GPR.sample_max_values)."""
        candidate_set = data_type_check(candidate_set)
        return super().sample_max_values(candidate_set, num_samples=num_samples, method=method, maximize=maximize,
                                         seed=seed)

    def noise_value(self):
        return self.likelihood.noise_covar.noise.detach() * self.y_std ** 2

    # ------------------------------------------------------------------------------------------
    def zeta_matrix(self, num_levels, embedding_dim: int, batch_shape=torch.Size()):
        """All level combinations (itertools.product order) and their concatenated one-hot encodings
        (gp_plus.py:1027-1073)."""
        if any([i == 1 for i in num_levels]):
            raise ValueError("Categorical variable has only one level!")
        if embedding_dim == 1:
            raise RuntimeWarning("1D latent variables are difficult to optimize!")
        for level in num_levels:
            if embedding_dim > level - 0:
                raise RuntimeWarning("The LV dimension can atmost be num_levels-1. Setting it to %s in place of %s"
                                     % (level - 1, min(embedding_dim, level - 1)))
        grids = torch.meshgrid(*[torch.arange(l) for l in num_levels], indexing="ij")
        perm = torch.stack([g.reshape(-1) for g in grids], dim=1).to(torch.int64)
        perm_dic = {str(row.tolist()): i for i, row in enumerate(perm)}
        one_hot = torch.cat([F.one_hot(perm[:, i], num_classes=int(num_levels[i])) for i in range(perm.shape[1])],
                            dim=1)
        return one_hot, perm, perm_dic

    def transform_categorical(self, x: torch.Tensor, perm_dict=[], zeta=[]):
        """One-hot rows of the level combinations in x (gp_plus.py:1077-1095); kept for API parity."""
        if x.dim() == 1:
            x = x.reshape(-1, 1)
        if self.training is False:
            x = torch.as_tensor(setlevels(x))
        try:
            index = [perm_dict[str(row.tolist())] for row in x.type(torch.int64)]
        except KeyError:
            raise ValueError("The categorical input (or source indices) are not defined properly. They should be "
                             "integer values starting from zero. To solve the issue, you can use the 'setlevels' "
                             "function, which is a preprocessing function.")
        return zeta[index, :]

    # ------------------------------------------------------------------------------------------
    # consumers of the batched prediction kernel (SURVEY 8f-2 / 8f-4)
    def Sobol(self, N=10000):
        """First-order and total Sobol sensitivity indices of the fitted emulator (models/gp_plus.py:1148-1224):
        Saltelli's A / B / AB_i design, (p + 2) * N predictions, all served by the batched predict kernel.

        Returns ``(S, ST)`` of shape [1, p].  Differences from the reference source, which cannot run as
        written: its ``normalize_sobol_sequence`` returns from inside the loop over categorical columns (only the
        first one is rounded, and a model without categorical inputs gets ``None``); here every categorical column
        is mapped to its levels.  The low-discrepancy points come from ``scipy.stats.qmc.Sobol(scramble=False)``
        (first point skipped, like ``sobol_seq.i4_sobol_generate``), since ``sobol_seq`` is not a dependency."""
        from scipy.stats.qmc import Sobol as _Sobol
        if N < 1e5:
            warnings.warn("Increase N for accuracy!")
        x = self.train_inputs[0].detach().double().cpu()
        p = x.shape[1]
        seq = torch.from_numpy(_Sobol(d=2 * p, scramble=False).random(N + 1)[1:])
        mins, maxs = x.min(dim=0)[0], x.max(dim=0)[0]
        parts = []
        for unit in (seq[:, p:], seq[:, :p]):
            pts = mins + (maxs - mins) * unit
            for k, col in enumerate(self._qual_cols):
                pts[:, col] = (unit[:, col] * (self.num_levels_per_var[k] - 1)).round()
            parts.append(pts)
        A, B = parts
        FA = self.predict(A, return_std=False).detach().cpu().numpy().reshape(-1, 1)
        FB = self.predict(B, return_std=False).detach().cpu().numpy().reshape(-1, 1)
        S, ST = np.zeros((p, 1)), np.zeros((p, 1))
        for i in range(p):
            ABi = A.clone()
            ABi[:, i] = B[:, i]
            Fi = self.predict(ABi, return_std=False).detach().cpu().numpy().reshape(-1, 1)
            S[i, :] = np.sum(FB * (Fi - FA), axis=0) / N
            ST[i, :] = np.sum((FA - Fi) ** 2, axis=0) / (2 * N)
        varY = np.var(np.concatenate([FA, FB]), axis=0)
        return (S / varY).T, (ST / varY).T

    def evaluation(self, Xtest, ytest, return_metrics: bool = False):
        """Test-set metrics of models/gp_plus.py:889-932: joint negative log predictive density per point (the
        full-covariance predictive of gpytorch.metrics.negative_log_predictive_density), MSE, MAE, RRMSE and the
        95 % interval score, in the original y units.

        The joint NLPD never forms the M x M predictive covariance: by the Schur-complement identity
        ``log p(y* | y) = log p(y, y*) - log p(y)`` it is the difference of two marginal-likelihood evaluations
        on the engine (training set alone, and training + test set with the test points' own noise groups)."""
        from tabulate import tabulate
        Xtest = data_type_check(Xtest).detach().double().cpu()
        ytest = data_type_check(ytest).detach().double().cpu().reshape(-1)
        self.eval()
        y_sc = (ytest - self.y_min) / self.y_std
        with torch.no_grad():
            mean, std = self.predict(Xtest, return_std=True, include_noise=True)
        mu = (mean - self.y_min) / self.y_std
        sd = std / self.y_std
        xtr = self.train_inputs[0].detach().double().cpu()
        if self._level_strides is not None:
            # the joint evaluation must see the test categories exactly as predict() does (eval-mode ranking)
            joint_levels = np.concatenate([self._level_index(xtr, True), self._level_index(Xtest, False)])
        else:
            joint_levels = None
        nll_train = self._joint_nll_with_levels(xtr, self.train_targets, None, True)
        nll_joint = self._joint_nll_with_levels(torch.cat([xtr, Xtest]), torch.cat([self.train_targets.double(), y_sc]),
                                                joint_levels, False)
        m = ytest.shape[0]
        nlpd = (nll_joint - nll_train) / m
        mse = torch.mean((mu - y_sc) ** 2) * self.y_std ** 2
        mae = torch.mean(torch.abs(mu - y_sc)) * torch.abs(self.y_std)
        lo, up = mu - 2.0 * sd, mu + 2.0 * sd  # MultivariateNormal.confidence_region: mean -/+ 2 std
        score = (up - lo) + (y_sc > up) * 2 / 0.05 * (y_sc - up) + (y_sc < lo) * 2 / 0.05 * (lo - y_sc)
        iscore = score.mean() * torch.abs(self.y_std)
        rrmse = torch.sqrt(mse / torch.var(ytest))
        table_data = [["Negative Log-Likelihood (NLL)", nlpd], ["Mean Squared Error (MSE)", mse],
                      ["Mean Absolute Error  (MAE)", mae], ["Relative Root Mean Square Error (RRMSE)", rrmse],
                      ["Interval Score (IS)", iscore]]
        print(tabulate(table_data, headers=["Metric", "Value"], tablefmt="fancy_grid", colalign=("left", "left")))
        if return_metrics:
            return {"NLL": float(nlpd), "MSE": float(mse), "MAE": float(mae), "RRMSE": float(rrmse),
                    "IS": float(iscore)}

    def _joint_nll_with_levels(self, x, y_scaled, levels, training: bool) -> float:
        from .. import _engine
        from .gpregression import get_default_device
        xc = x.detach().double().cpu()
        cols = self._quant_columns()
        qk = self._quant_kernel() if len(cols) > 0 else None
        table = self._latent_table()
        n_mean, _ = self._mean_layout()
        if levels is None:
            levels = self._level_index(xc, training)
        eng = _engine.Engine(
            xq=xc[:, cols].numpy() if qk is not None else None, y=y_scaled.detach().double().cpu().numpy(),
            kernel=qk.family if qk is not None else _engine.KERNEL_EXPSQ, level_idx=levels,
            n_combo=0 if table is None else int(table.shape[0]), dz=0 if table is None else int(table.shape[1]),
            noise_idx=self._noise_index(xc), n_noise=int(self.likelihood.noise_covar.raw_noise.numel()),
            mean_idx=self._mean_index(xc), n_mean=n_mean, device=get_default_device())
        try:
            return float(eng.mll_grad(self._hyper_numpy(), want_grad=False)["nll"])
        finally:
            eng.close()


    def score(self, Xtest, ytest, plot_MSE=True, title=None, seperate_levels=False):
        """MSE of the predictive mean and the estimated noise, printed as the reference does (gp_plus.py:634-666).
        The parity plot is drawn only when matplotlib is installed."""
        Xtest = data_type_check(Xtest)
        ytest = data_type_check(ytest).reshape(-1)
        ypred = self.predict(Xtest, return_std=False)
        mse = ((ytest - ypred) ** 2).mean()
        noise = self.noise_value()
        print("################MSE######################")
        print(f"MSE = {mse:.5f}")
        print("################Noise####################")
        print(f"The estimated noise parameter (varaince) is {noise}")
        print(f"The estimated noise std is {np.sqrt(noise.cpu())}")
        print("#########################################")
        if plot_MSE:
            try:
                import matplotlib.pyplot as plt
            except ImportError:
                plt = None
            if plt is not None:
                plt.figure(figsize=(8, 6))
                plt.plot(ytest.numpy(), ypred.numpy(), "ro", label="Data")
                plt.plot(ytest.numpy(), ytest.numpy(), "b", label="MSE = " + str(np.round(float(mse), 3)))
                plt.xlabel(r"Y_True")
                plt.ylabel(r"Y_predict")
                plt.legend()
                if title is not None:
                    plt.title(title)
        if seperate_levels and len(self._qual_cols) > 0:
            for level in range(self.num_levels_per_var[0]):
                rows = torch.where(Xtest[:, self._qual_cols[0]] == level)[0]
                self.score(Xtest[rows, ...], ytest[rows], plot_MSE=plot_MSE,
                           title="results Only Source " + str(level), seperate_levels=False)
        return ypred

    def get_params(self, name=None):
        """Raw parameters by their state-dict names, or one of 'Mean' / 'Sigma' / 'Noise' / 'Omega'
        (gp_plus.py:962-982)."""
        params = {n: value for n, value in self.named_parameters()}
        print("###################Parameters###########################")
        if name is None:
            print(params)
            return params
        key = {"Mean": "mean_module.constant", "Sigma": "covar_module.raw_outputscale",
               "Noise": "likelihood.noise_covar.raw_noise"}.get(name)
        if name == "Omega":
            ls = [n for n, v in params.items() if "raw_lengthscale" in n]
            ard = [n for n in ls if params[n].numel() > 1]  # the reference picks the ARD one; 1-D inputs have none
            key = (ard or ls or [None])[-1]
        if key is None:
            raise KeyError(name)
        print(params[key])
        return params[key]

    def get_latent_space(self):
        if len(self.qual_kernel_columns) == 0:
            raise RuntimeError("No categorical Variable, No latent positions")
        with torch.no_grad():
            dtype = self.covar_module.raw_outputscale.dtype
            if self.embedding_type == "probabilistic":
                return self._sampled_latent_tables(dtype).detach()
            return self._latent_map(self.zeta[-1].to(dtype)).detach()


class Linear_MAP(nn.Linear):
    """Bias-free linear latent map z = zeta A^T (gp_plus.py:1456-1461)."""

    def forward(self, input, transform=lambda x: x):
        return F.linear(input, transform(self.weight), self.bias)


class Linear_VAE(_CompatModule):
    """Affine layer of the variational encoder (gp_plus.py:1302-1341): weight / bias registered under
    ``<name>weight`` / ``<name>bias`` with N(0, 0.2) / N(0, 0.05) priors; evaluated in float64."""

    def __init__(self, in_features: int, out_features: int, bias: bool = True, name=None):
        super().__init__()
        self.in_features, self.out_features, self.name = in_features, out_features, str(name)
        self.register_parameter(self.name + "weight", nn.Parameter(torch.empty((out_features, in_features))))
        self.register_prior(self.name + "prior_m_weight_fci", NormalPrior(0.0, 0.2), self.name + "weight")
        if bias:
            self.register_parameter(self.name + "bias", nn.Parameter(torch.empty(out_features)))
            self.register_prior(self.name + "prior_m_bias_fci", NormalPrior(0.0, 0.05), self.name + "bias")
        else:
            self.register_parameter("bias", None)
        w = getattr(self, self.name + "weight")
        nn.init.kaiming_uniform_(w, a=math.sqrt(5))
        b = getattr(self, self.name + "bias", None)
        if b is not None:
            fan_in, _ = nn.init._calculate_fan_in_and_fan_out(w)
            bound = 1 / math.sqrt(fan_in) if fan_in > 0 else 0
            nn.init.uniform_(b, -bound, bound)

    def forward(self, input):
        return F.linear(input.double(), getattr(self, self.name + "weight").double(),
                        getattr(self, self.name + "bias").double())


class Variational_Encoder(_CompatModule):
    """(one-hot row, epsilon) -> 2-D latent position (gp_plus.py:1373-1413): the network outputs
    (L22, L21, L11, mu2, mu1) and the position is mu + L epsilon with |.| on the diagonal of L.  With hidden layers the
    FIRST layer has no activation (as in the reference), the others are tanh."""

    def __init__(self, input_size, num_classes, layers):
        super().__init__()
        self.hidden_num = len(layers)
        if self.hidden_num > 0:
            self.fci = Linear_VAE(input_size, layers[0], bias=True, name="fci")
            for i in range(1, self.hidden_num):
                setattr(self, "h" + str(i), Linear_VAE(layers[i - 1], layers[i], bias=True, name="h" + str(i)))
            self.fce = Linear_VAE(layers[-1], num_classes, bias=True, name="fce")
        else:
            self.fci = Linear_VAE(input_size, num_classes, bias=True, name="fci")

    def forward(self, x, epsilon):
        if self.hidden_num > 0:
            x = self.fci(x)
            for i in range(1, self.hidden_num):
                x = torch.tanh(getattr(self, "h" + str(i))(x))
            output = self.fce(x)
        else:
            output = self.fci(x)
        e1, e2 = epsilon[:, 0:1], epsilon[:, 1:2]
        L22, L21, L11, mu2, mu1 = (output[:, k:k + 1] for k in range(5))
        x1 = mu1 + 1 * torch.abs(L11) * e1
        x2 = mu2 + 1 * L21 * e1 + 1 * torch.abs(L22) * e2
        return torch.cat((x1, x2), 1)


class FFNN(nn.Module):
    """Latent map: a bias-free linear layer, or a tanh MLP when hidden ``layers`` are given.  Weights are
    registered on the owning model (so they pack into theta first) with N(0,1) priors (gp_plus.py:1227-1265)."""

    def __init__(self, owner, input_size, num_classes, layers, name):
        super().__init__()
        self.hidden_num = len(layers)
        if self.hidden_num > 0:
            self.fci = nn.Linear(input_size, layers[0], bias=False)
            owner.register_parameter(str(name) + "fci", self.fci.weight)
            owner.register_prior(name="latent_prior_fci", prior=NormalPrior(0.0, 1),
                                 param_or_closure=str(name) + "fci")
            for i in range(1, self.hidden_num):
                setattr(self, "h" + str(i), nn.Linear(layers[i - 1], layers[i], bias=False))
                owner.register_parameter(str(name) + "h" + str(i), getattr(self, "h" + str(i)).weight)
                owner.register_prior(name="latent_prior" + str(i), prior=NormalPrior(0.0, 1),
                                     param_or_closure=str(name) + "h" + str(i))
            self.fce = nn.Linear(layers[-1], num_classes, bias=False)
            owner.register_parameter(str(name) + "fce", self.fce.weight)
            owner.register_prior(name="latent_prior_fce", prior=NormalPrior(0.0, 1),
                                 param_or_closure=str(name) + "fce")
        else:
            self.fci = Linear_MAP(input_size, num_classes, bias=False)
            owner.register_parameter(name, self.fci.weight)
            owner.register_prior(name="latent_prior_" + name, prior=NormalPrior(0, 1), param_or_closure=name)

    def forward(self, x, transform=lambda x: x):
        if self.hidden_num > 0:
            x = torch.tanh(self.fci(x))
            for i in range(1, self.hidden_num):
                x = torch.tanh(getattr(self, "h" + str(i))(x))
            return self.fce(x)
        return self.fci(x, transform)
