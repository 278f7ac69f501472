"""ctypes binding of ``libgpplus_b200.so`` -- the C-ABI declared in ``include/gpplus_b200.h``.

The library is the only compute path of this package: if it is missing, fails to load, or no
B200 is visible, every call raises; nothing here falls back to torch or numpy arithmetic.
"""
from __future__ import annotations

import ctypes as C
import os
import threading
from typing import Dict, Sequence

import numpy as np

GPP_OK, GPP_ERR_NOT_PD, GPP_ERR_NAN, GPP_ERR_ARG, GPP_ERR_CUDA = 0, 1, 2, 3, -1
KERNEL_EXPSQ, KERNEL_MATERN32, KERNEL_MATERN52 = 0, 1, 2
ACQ_HF, ACQ_LF, ACQ_EI = 0, 1, 2
MAX_DQ, MAX_DZ = 32, 4
MAX_JOINT = 16384  # GPP_MAX_JOINT: candidates of one gpp_predict_joint / gpp_sample_posterior call
MAX_QBATCH = 128  # GPP_MAX_QBATCH: points per t-batch of gpp_posterior_qbatch / gpp_posterior_qbatch_grad
QACQ_EI, QACQ_NEI, QACQ_UCB = 0, 1, 2  # GPP_QACQ_*: utilities of gpp_acq_qbatch
MAX_MC_SAMPLES = 65536  # GPP_MAX_MC_SAMPLES: base-sample rows of one gpp_acq_qbatch call
MAX_IPV_POINTS = 16384  # GPP_MAX_IPV_POINTS: integration points of one gpp_ipv_points call

LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib", "libgpplus_b200.so")

EXPORTS = (
    "gpp_version", "gpp_device_count", "gpp_last_error", "gpp_launch_count", "gpp_create", "gpp_destroy", "gpp_pool_clear",
    "gpp_mll_grad",
    "gpp_get_timings", "gpp_get_stats", "gpp_covariance", "gpp_fetch", "gpp_factorize", "gpp_predict", "gpp_predict_grad",
    "gpp_predict_joint", "gpp_sample_posterior", "gpp_posterior_qbatch", "gpp_posterior_qbatch_grad", "gpp_acq_qbatch",
    "gpp_ipv_points", "gpp_nipv_qbatch", "gpp_kg_qbatch", "gpp_gibbon_qbatch", "gpp_max_value_quartiles",
    "gpp_acq_argmax",
    "gpp_probe_dgemm", "gpp_probe_i8", "gpp_set_fp64_mode", "gpp_get_fp64_mode", "gpp_set_theta_layout", "gpp_objective", "gpp_objective_enqueue", "gpp_objective_collect",
)

PRIOR_NORMAL, PRIOR_LOGNORMAL_OS, PRIOR_HORSESHOE, PRIOR_MOLLIFIED, PRIOR_CONST = 0, 1, 2, 3, 4


class NotPSDError(RuntimeError):
    """K_y not positive definite after the jitter ladder (gpytorch.utils.errors.NotPSDError)."""


class NanError(RuntimeError):
    """NaN in K_y / the likelihood (gpytorch.utils.errors.NanError)."""


class EngineError(RuntimeError):
    pass


_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int32)


class _Problem(C.Structure):
    _fields_ = [("n", C.c_int64), ("dq", C.c_int32), ("dz", C.c_int32), ("n_combo", C.c_int32),
                ("n_noise", C.c_int32), ("n_mean", C.c_int32), ("kernel", C.c_int32),
                ("xq", _dp), ("y", _dp), ("level_idx", _ip), ("noise_idx", _ip), ("mean_idx", _ip),
                ("n_pass", C.c_int32)]


class _Hyper(C.Structure):
    _fields_ = [("w", _dp), ("z", _dp), ("sigma_f2", C.c_double), ("noise", _dp), ("beta", _dp)]


class _MllResult(C.Structure):
    _fields_ = [("nll", C.c_double), ("logdet", C.c_double), ("quad", C.c_double), ("jitter", C.c_double),
                ("d_sigma_f2", C.c_double), ("d_w", _dp), ("d_z", _dp), ("d_noise", _dp), ("d_beta", _dp)]


class _Prior(C.Structure):
    _fields_ = [("kind", C.c_int32), ("off", C.c_int32), ("len", C.c_int32), ("a", _dp), ("b", _dp), ("c", _dp)]


class _ThetaLayout(C.Structure):
    _fields_ = [("p", C.c_int32), ("off_latent", C.c_int32), ("n_onehot", C.c_int32), ("zeta", _dp),
                ("latent_const", _dp), ("latent_ls", C.c_double), ("off_noise", C.c_int32), ("noise_const", _dp),
                ("noise_lb", C.c_double), ("off_os", C.c_int32), ("os_const", C.c_double), ("off_ls", C.c_int32),
                ("ls_const", _dp), ("ls_kind", C.c_int32), ("w_num", C.c_double), ("off_mean", _ip),
                ("mean_const", _dp), ("n_priors", C.c_int32), ("priors", C.POINTER(_Prior))]


class _Timings(C.Structure):
    _fields_ = [("covariance", C.c_float), ("cholesky", C.c_float), ("trtri", C.c_float), ("solve", C.c_float),
                ("lauum", C.c_float), ("gradient", C.c_float), ("total", C.c_float)]


class _Stats(C.Structure):
    _fields_ = [("evaluations", C.c_int64), ("factorizations", C.c_int64), ("jitter_retries", C.c_int64),
                ("early_outs", C.c_int64)]


_lib = None
_lib_lock = threading.Lock()


def load_library():
    """Load the shared library (once).  Raises EngineError if it has not been built."""
    global _lib
    with _lib_lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise EngineError(
                "gpplus_b200: %s is missing. Build it with `python __graft_entry__.py build` "
                "(nvcc -gencode arch=compute_100a,code=sm_100a). There is no CPU fallback." % LIB_PATH)
        lib = C.CDLL(LIB_PATH)
        lib.gpp_version.restype = C.c_int
        lib.gpp_device_count.restype = C.c_int
        lib.gpp_last_error.restype = C.c_char_p
        lib.gpp_launch_count.restype = C.c_longlong
        lib.gpp_create.argtypes = [C.POINTER(_Problem), C.c_int, C.POINTER(C.c_void_p)]
        lib.gpp_create.restype = C.c_int
        lib.gpp_destroy.argtypes = [C.c_void_p]
        lib.gpp_destroy.restype = None
        lib.gpp_pool_clear.argtypes = []
        lib.gpp_pool_clear.restype = None
        lib.gpp_mll_grad.argtypes = [C.c_void_p, C.POINTER(_Hyper), C.c_int, C.POINTER(_MllResult)]
        lib.gpp_mll_grad.restype = C.c_int
        lib.gpp_get_timings.argtypes = [C.c_void_p, C.POINTER(_Timings)]
        lib.gpp_get_timings.restype = C.c_int
        lib.gpp_get_stats.argtypes = [C.c_void_p, C.POINTER(_Stats)]
        lib.gpp_get_stats.restype = C.c_int
        lib.gpp_covariance.argtypes = [C.c_void_p, C.POINTER(_Hyper), C.c_void_p]
        lib.gpp_covariance.restype = C.c_int
        lib.gpp_fetch.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        lib.gpp_fetch.restype = C.c_int
        lib.gpp_factorize.argtypes = [C.c_void_p, C.POINTER(_Hyper)]
        lib.gpp_factorize.restype = C.c_int
        lib.gpp_predict.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                    C.c_double, C.c_void_p, C.c_void_p]
        lib.gpp_predict.restype = C.c_int
        lib.gpp_predict_grad.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_int, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.gpp_predict_grad.restype = C.c_int
        lib.gpp_predict_joint.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_int, C.c_void_p, C.c_void_p]
        lib.gpp_predict_joint.restype = C.c_int
        lib.gpp_sample_posterior.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                             C.c_int, C.c_int64, C.c_void_p, C.c_void_p, C.POINTER(C.c_double)]
        lib.gpp_sample_posterior.restype = C.c_int
        lib.gpp_posterior_qbatch.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                             C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
        lib.gpp_posterior_qbatch.restype = C.c_int
        lib.gpp_posterior_qbatch_grad.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p,
                                                  C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.gpp_posterior_qbatch_grad.restype = C.c_int
        lib.gpp_acq_qbatch.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_int, C.c_int, C.c_int32, C.c_double, C.c_double, C.c_int,
                                       C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.gpp_acq_qbatch.restype = C.c_int
        lib.gpp_ipv_points.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
        lib.gpp_ipv_points.restype = C.c_int
        lib.gpp_nipv_qbatch.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.c_void_p]
        lib.gpp_nipv_qbatch.restype = C.c_int
        lib.gpp_kg_qbatch.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.gpp_kg_qbatch.restype = C.c_int
        lib.gpp_gibbon_qbatch.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_void_p]
        lib.gpp_gibbon_qbatch.restype = C.c_int
        lib.gpp_max_value_quartiles.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                                C.c_void_p]
        lib.gpp_max_value_quartiles.restype = C.c_int
        lib.gpp_acq_argmax.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_double,
                                       C.c_double, C.c_double, C.c_double, C.c_void_p, _dp, C.POINTER(C.c_int64)]
        lib.gpp_acq_argmax.restype = C.c_int
        lib.gpp_probe_dgemm.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float)]
        lib.gpp_probe_dgemm.restype = C.c_int
        lib.gpp_probe_i8.argtypes = [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_double)]
        lib.gpp_probe_i8.restype = C.c_int
        lib.gpp_set_fp64_mode.argtypes = [C.c_int]
        lib.gpp_set_fp64_mode.restype = C.c_int
        lib.gpp_get_fp64_mode.argtypes = [C.c_void_p]
        lib.gpp_get_fp64_mode.restype = C.c_int
        lib.gpp_set_theta_layout.argtypes = [C.c_void_p, C.POINTER(_ThetaLayout)]
        lib.gpp_set_theta_layout.restype = C.c_int
        lib.gpp_objective.argtypes = [C.c_void_p, C.c_void_p, C.c_int, _dp, C.c_void_p, C.POINTER(_MllResult)]
        lib.gpp_objective.restype = C.c_int
        lib.gpp_objective_enqueue.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        lib.gpp_objective_enqueue.restype = C.c_int
        lib.gpp_objective_collect.argtypes = [C.c_void_p, _dp, C.c_void_p, C.POINTER(_MllResult)]
        lib.gpp_objective_collect.restype = C.c_int
        _lib = lib
        return lib


def launch_count() -> int:
    """CUDA kernels launched by the library in this process so far."""
    return int(load_library().gpp_launch_count())


def pool_clear():
    """Free every parked engine handle (see gpp_destroy in include/gpplus_b200.h)."""
    load_library().gpp_pool_clear()


def device_count() -> int:
    return int(load_library().gpp_device_count())


def _raise(rc: int, where: str):
    msg = load_library().gpp_last_error().decode("utf-8", "replace")
    if rc == GPP_ERR_NOT_PD:
        raise NotPSDError(msg or "Matrix not positive definite after repeatedly adding jitter up to 1e-06.")
    if rc == GPP_ERR_NAN:
        raise NanError(msg or "NaN in the covariance matrix")
    if rc == GPP_ERR_ARG:
        raise ValueError("%s: %s" % (where, msg))
    raise EngineError("%s failed (status %d): %s" % (where, rc, msg))


def _f64(a, shape=None):
    a = np.ascontiguousarray(np.asarray(a, dtype=np.float64))
    if shape is not None:
        a = a.reshape(shape)
    return a


def _i32(a, n):
    if a is None:
        return None
    a = np.ascontiguousarray(np.asarray(a).astype(np.int32, copy=False)).reshape(n)
    return a


def _ptr(a):
    """void* of a numpy array, a torch tensor (host or cuda:<this device>) or None."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return C.c_void_p(a.ctypes.data)
    return C.c_void_p(int(a.data_ptr()))  # torch tensor, contiguous by contract


class Engine:
    """One training set resident on one GPU (``gpp_handle``).  Not thread-safe; use one per in-flight restart."""

    def __init__(self, xq, y, kernel: int, level_idx=None, n_combo: int = 0, dz: int = 0, noise_idx=None,
                 n_noise: int = 1, mean_idx=None, n_mean: int = 1, device: int = 0, n_pass: int = 1):
        lib = load_library()
        y = _f64(y).reshape(-1)
        n = y.shape[0]
        xq = _f64(xq).reshape(n, -1) if xq is not None and np.size(xq) else np.zeros((n, 0))
        self.n, self.dq, self.dz = n, xq.shape[1], int(dz)
        self.n_combo, self.n_noise, self.n_mean, self.kernel = int(n_combo), int(n_noise), int(n_mean), int(kernel)
        self.device = int(device)
        self.n_pass = max(1, int(n_pass))
        self._keep = (xq, y, _i32(level_idx, n), _i32(noise_idx, n), _i32(mean_idx, n))
        p = _Problem()
        p.n, p.dq, p.dz, p.n_combo = n, self.dq, self.dz, self.n_combo
        p.n_noise, p.n_mean, p.kernel = self.n_noise, self.n_mean, self.kernel
        p.n_pass = self.n_pass
        p.xq = xq.ctypes.data_as(_dp) if self.dq > 0 else None
        p.y = y.ctypes.data_as(_dp)
        for name, arr in zip(("level_idx", "noise_idx", "mean_idx"), self._keep[2:]):
            setattr(p, name, arr.ctypes.data_as(_ip) if arr is not None else None)
        h = C.c_void_p()
        rc = lib.gpp_create(C.byref(p), self.device, C.byref(h))
        if rc != GPP_OK:
            _raise(rc, "gpp_create")
        self._h = h
        self._lib = lib

    def close(self):
        if getattr(self, "_h", None):
            self._lib.gpp_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- hyper-parameters -------------------------------------------------------------------
    def _hyper(self, hyper: Dict):
        w = _f64(hyper.get("w", np.zeros(0))).reshape(-1)
        if w.shape[0] != self.dq:
            raise ValueError("hyper['w'] must have %d entries" % self.dq)
        z = None
        if self.dz > 0:
            z = _f64(hyper["z"]).reshape(-1)
            if z.shape[0] != self.n_pass * self.n_combo * self.dz:
                raise ValueError("hyper['z'] must be [n_combo, dz] (or [n_pass, n_combo, dz])")
        noise = _f64(hyper["noise"]).reshape(-1)
        if noise.shape[0] != self.n_noise:
            raise ValueError("hyper['noise'] must have %d entries" % self.n_noise)
        beta = None
        if self.n_mean > 0:
            beta = _f64(hyper["beta"]).reshape(-1)
            if beta.shape[0] != self.n_mean:
                raise ValueError("hyper['beta'] must have %d entries" % self.n_mean)
        hy = _Hyper()
        hy.w = w.ctypes.data_as(_dp) if self.dq > 0 else None
        hy.z = z.ctypes.data_as(_dp) if z is not None else None
        hy.sigma_f2 = float(hyper["sigma_f2"])
        hy.noise = noise.ctypes.data_as(_dp)
        hy.beta = beta.ctypes.data_as(_dp) if beta is not None else None
        return hy, (w, z, noise, beta)

    # -- MLL ----------------------------------------------------------------------------------
    def mll_grad(self, hyper: Dict, want_grad: bool = True) -> Dict:
        hy, keep = self._hyper(hyper)
        res = _MllResult()
        d_w = np.zeros(max(self.dq, 1))
        d_z = np.zeros(max(self.n_pass * self.n_combo * self.dz, 1))
        d_noise = np.zeros(self.n_noise)
        d_beta = np.zeros(max(self.n_mean, 1))
        res.d_w, res.d_z = d_w.ctypes.data_as(_dp), d_z.ctypes.data_as(_dp)
        res.d_noise, res.d_beta = d_noise.ctypes.data_as(_dp), d_beta.ctypes.data_as(_dp)
        rc = self._lib.gpp_mll_grad(self._h, C.byref(hy), 1 if want_grad else 0, C.byref(res))
        del keep
        if rc != GPP_OK:
            _raise(rc, "gpp_mll_grad")
        out = {"nll": res.nll, "logdet": res.logdet, "quad": res.quad, "jitter": res.jitter}
        if want_grad:
            out["d_sigma_f2"] = res.d_sigma_f2
            out["d_w"] = d_w[: self.dq].copy()
            out["d_noise"] = d_noise
            if self.dz > 0:
                out["d_z"] = d_z.reshape(self.n_combo, self.dz) if self.n_pass == 1 else \
                    d_z.reshape(self.n_pass, self.n_combo, self.dz)
            if self.n_mean > 0:
                out["d_beta"] = d_beta[: self.n_mean]
        return out

    # -- objective in raw theta (the whole body of MLLObjective.fun in one GIL-free call) -----------------
    def set_theta_layout(self, spec: Dict):
        """``spec``: the dictionary produced by ``FastObjective.layout_spec()`` (optim/_fast_objective.py)."""
        keep = []

        def arr(a):
            if a is None:
                return None
            a = _f64(a).reshape(-1)
            keep.append(a)
            return a.ctypes.data_as(_dp)

        lay = _ThetaLayout()
        lay.p = int(spec["p"])
        lay.off_latent = int(spec.get("off_latent", -1))
        lay.n_onehot = int(spec.get("n_onehot", 0))
        lay.zeta = arr(spec.get("zeta"))
        lay.latent_const = arr(spec.get("latent_const"))
        lay.latent_ls = float(spec.get("latent_ls", 1.0))
        lay.off_noise = int(spec["off_noise"])
        lay.noise_const = arr(spec.get("noise_const"))
        lay.noise_lb = float(spec["noise_lb"])
        lay.off_os = int(spec["off_os"])
        lay.os_const = float(spec.get("os_const", 0.0))
        lay.off_ls = int(spec.get("off_ls", -1))
        lay.ls_const = arr(spec.get("ls_const"))
        lay.ls_kind = int(spec.get("ls_kind", 0))
        lay.w_num = float(spec.get("w_num", 0.5))
        om = np.ascontiguousarray(np.asarray(spec.get("off_mean", []), dtype=np.int32))
        keep.append(om)
        lay.off_mean = om.ctypes.data_as(_ip) if om.size else None
        lay.mean_const = arr(spec.get("mean_const")) if om.size else None
        pri = spec.get("priors", [])
        parr = (_Prior * max(len(pri), 1))()
        for i, (kind, off, length, a, b, c) in enumerate(pri):
            parr[i].kind, parr[i].off, parr[i].len = int(kind), int(off), int(length)
            parr[i].a, parr[i].b, parr[i].c = arr(a), arr(b), arr(c)
        lay.n_priors = len(pri)
        lay.priors = parr
        rc = self._lib.gpp_set_theta_layout(self._h, C.byref(lay))
        del keep
        if rc != GPP_OK:
            _raise(rc, "gpp_set_theta_layout")
        self._p = lay.p
        self._grad_buf = np.zeros(lay.p)
        self._val_buf = C.c_double()

    def objective(self, theta, want_grad: bool = True):
        """(neg log posterior, gradient) at raw ``theta``; the gradient array is freshly allocated."""
        th = np.ascontiguousarray(theta, dtype=np.float64)
        if th.shape[0] != self._p:
            raise ValueError("theta must have %d entries" % self._p)
        grad = np.empty(self._p) if want_grad else None
        rc = self._lib.gpp_objective(self._h, th.ctypes.data, 1 if want_grad else 0, C.byref(self._val_buf),
                                     grad.ctypes.data if want_grad else None, None)
        if rc != GPP_OK:
            _raise(rc, "gpp_objective")
        if want_grad:
            return self._val_buf.value, grad
        return self._val_buf.value

    def objective_enqueue(self, theta, want_grad: bool = True):
        """Issue ``objective(theta)`` on this handle's stream without waiting (pair with ``objective_collect``)."""
        th = np.ascontiguousarray(theta, dtype=np.float64)
        if th.shape[0] != self._p:
            raise ValueError("theta must have %d entries" % self._p)
        self._pending_theta = th  # keep the buffer alive until the call returns (it is copied inside)
        rc = self._lib.gpp_objective_enqueue(self._h, th.ctypes.data, 1 if want_grad else 0)
        if rc != GPP_OK:
            _raise(rc, "gpp_objective_enqueue")

    def objective_collect(self, grad_out=None):
        """Wait for the enqueued evaluation; returns the value and writes the gradient into ``grad_out`` (length p).
        Raises NotPSDError / NanError exactly like ``objective``."""
        rc = self._lib.gpp_objective_collect(self._h, C.byref(self._val_buf),
                                             grad_out.ctypes.data if grad_out is not None else None, None)
        if rc != GPP_OK:
            _raise(rc, "gpp_objective_collect")
        return self._val_buf.value

    def timings(self) -> Dict[str, float]:
        t = _Timings()
        rc = self._lib.gpp_get_timings(self._h, C.byref(t))
        if rc != GPP_OK:
            _raise(rc, "gpp_get_timings")
        return {k: float(getattr(t, k)) for k, _ in _Timings._fields_}

    def fp64_mode(self) -> int:
        """FP64_DMMA or FP64_INT8: the arithmetic this handle uses for the O(N^3) stages (gpp_get_fp64_mode)."""
        return int(self._lib.gpp_get_fp64_mode(self._h))

    def stats(self) -> Dict[str, int]:
        st = _Stats()
        rc = self._lib.gpp_get_stats(self._h, C.byref(st))
        if rc != GPP_OK:
            _raise(rc, "gpp_get_stats")
        return {k: int(getattr(st, k)) for k, _ in _Stats._fields_}

    def covariance(self, hyper: Dict) -> np.ndarray:
        hy, keep = self._hyper(hyper)
        out = np.empty((self.n, self.n))
        rc = self._lib.gpp_covariance(self._h, C.byref(hy), _ptr(out))
        del keep
        if rc != GPP_OK:
            _raise(rc, "gpp_covariance")
        return out

    def fetch(self, which: str) -> np.ndarray:
        code = {"L": 0, "Linv": 1, "Kinv": 2, "alpha": 3, "Kinv_diag": 4}[which]
        out = np.empty(self.n if code >= 3 else (self.n, self.n))
        rc = self._lib.gpp_fetch(self._h, code, _ptr(out))
        if rc != GPP_OK:
            _raise(rc, "gpp_fetch")
        return out

    # -- prediction -------------------------------------------------------------------------
    def factorize(self, hyper: Dict):
        hy, keep = self._hyper(hyper)
        rc = self._lib.gpp_factorize(self._h, C.byref(hy))
        del keep
        if rc != GPP_OK:
            _raise(rc, "gpp_factorize")

    def predict(self, xq, level_idx=None, noise_idx=None, mean_idx=None, include_noise: bool = False,
                min_var: float = 1e-10, out_mean=None, out_var=None):
        """xq / index arrays may be numpy (host) or contiguous torch tensors on this engine's GPU."""
        xq, m, level_idx, noise_idx, mean_idx = self._candidates(xq, level_idx, noise_idx, mean_idx)
        mean = np.empty(m) if out_mean is None else out_mean
        var = np.empty(m) if out_var is None else out_var
        rc = self._lib.gpp_predict(self._h, m, _ptr(xq), _ptr(level_idx), _ptr(noise_idx), _ptr(mean_idx),
                                   1 if include_noise else 0, float(min_var), _ptr(mean), _ptr(var))
        if rc != GPP_OK:
            _raise(rc, "gpp_predict")
        return mean, var

    def predict_grad(self, xq, level_idx=None, noise_idx=None, mean_idx=None, include_noise: bool = False,
                     min_var: float = 1e-10, out_mean=None, out_var=None, out_d_mean=None, out_d_var=None):
        """``predict`` plus the derivatives of the scaled mean and of the clamped variance with respect to the
        quantitative inputs: returns ``(mean [m], var [m], d_mean [m, dq], d_var [m, dq])``.  Inputs and output
        buffers as for ``predict``."""
        xq, m, level_idx, noise_idx, mean_idx = self._candidates(xq, level_idx, noise_idx, mean_idx)
        mean = np.empty(m) if out_mean is None else out_mean
        var = np.empty(m) if out_var is None else out_var
        d_mean = np.empty((m, self.dq)) if out_d_mean is None else out_d_mean
        d_var = np.empty((m, self.dq)) if out_d_var is None else out_d_var
        rc = self._lib.gpp_predict_grad(self._h, m, _ptr(xq), _ptr(level_idx), _ptr(noise_idx), _ptr(mean_idx),
                                        1 if include_noise else 0, float(min_var), _ptr(mean), _ptr(var),
                                        _ptr(d_mean), _ptr(d_var))
        if rc != GPP_OK:
            _raise(rc, "gpp_predict_grad")
        return mean, var, d_mean, d_var

    def _candidates(self, xq, level_idx, noise_idx, mean_idx):
        if isinstance(xq, np.ndarray) or not hasattr(xq, "data_ptr"):
            xq = _f64(xq)
            m = xq.shape[0] if xq.ndim == 2 else (xq.size // max(self.dq, 1))
            return xq, m, _i32(level_idx, m), _i32(noise_idx, m), _i32(mean_idx, m)
        return xq, int(xq.shape[0]), level_idx, noise_idx, mean_idx

    def predict_joint(self, xq, level_idx=None, noise_idx=None, mean_idx=None, include_noise: bool = False,
                      out_mean=None, out_cov=None):
        """Predictive mean [m] (bitwise ``predict``'s) and the full, unclamped predictive covariance [m, m] in scaled y
        units (gpp_predict_joint).  Inputs and output buffers as for ``predict``; m <= MAX_JOINT."""
        xq, m, level_idx, noise_idx, mean_idx = self._candidates(xq, level_idx, noise_idx, mean_idx)
        mean = np.empty(m) if out_mean is None else out_mean
        cov = np.empty((m, m)) if out_cov is None else out_cov
        rc = self._lib.gpp_predict_joint(self._h, m, _ptr(xq), _ptr(level_idx), _ptr(noise_idx), _ptr(mean_idx),
                                         1 if include_noise else 0, _ptr(mean), _ptr(cov))
        if rc != GPP_OK:
            _raise(rc, "gpp_predict_joint")
        return mean, cov

    def sample_posterior(self, xq, base_samples, level_idx=None, noise_idx=None, mean_idx=None,
                         include_noise: bool = False, out=None):
        """Draws ``mean + base_samples L^T`` from the joint posterior with ``L L^T = cov + jitter I``
        (gpp_sample_posterior): returns ``(samples [S, m], jitter)``.  ``base_samples`` [S, m] may live on the host or
        on this engine's GPU, like the other inputs."""
        xq, m, level_idx, noise_idx, mean_idx = self._candidates(xq, level_idx, noise_idx, mean_idx)
        if isinstance(base_samples, np.ndarray) or not hasattr(base_samples, "data_ptr"):
            base_samples = _f64(base_samples)
        if len(base_samples.shape) != 2 or int(base_samples.shape[1]) != m:
            raise ValueError("sample_posterior: base_samples must have shape [S, %d], got %s"
                             % (m, tuple(base_samples.shape)))
        s = int(base_samples.shape[0])
        samples = np.empty((s, m)) if out is None else out
        jit = C.c_double(0.0)
        rc = self._lib.gpp_sample_posterior(self._h, m, _ptr(xq), _ptr(level_idx), _ptr(noise_idx), _ptr(mean_idx),
                                            1 if include_noise else 0, s, _ptr(base_samples), _ptr(samples),
                                            C.byref(jit))
        if rc != GPP_OK:
            _raise(rc, "gpp_sample_posterior")
        return samples, float(jit.value)

    @staticmethod
    def _tbatches(m, q, caller, q_name="q"):
        """(b, q) of m rows split into t-batches of q consecutive rows; ValueError naming ``caller`` otherwise."""
        q = int(q)
        if q < 1 or m % q:
            raise ValueError("%s: %d rows do not split into t-batches of %s = %d" % (caller, m, q_name, q))
        return m // q, q

    def posterior_qbatch(self, xq, q, level_idx=None, noise_idx=None, mean_idx=None, include_noise: bool = False,
                         out_mean=None, out_cov=None):
        """Mean [b, q] (bitwise ``predict``'s) and joint covariance [b, q, q] of b t-batches of q consecutive rows of
        ``xq`` in scaled y units (gpp_posterior_qbatch): each block exactly symmetric and not clamped.  Inputs and
        output buffers as for ``predict``; q <= MAX_QBATCH."""
        xq, m, level_idx, noise_idx, mean_idx = self._candidates(xq, level_idx, noise_idx, mean_idx)
        b, q = self._tbatches(m, q, "posterior_qbatch")
        mean = np.empty((b, q)) if out_mean is None else out_mean
        cov = np.empty((b, q, q)) if out_cov is None else out_cov
        rc = self._lib.gpp_posterior_qbatch(self._h, b, q, _ptr(xq), _ptr(level_idx), _ptr(noise_idx), _ptr(mean_idx),
                                            1 if include_noise else 0, _ptr(mean), _ptr(cov))
        if rc != GPP_OK:
            _raise(rc, "gpp_posterior_qbatch")
        return mean, cov

    def posterior_qbatch_grad(self, xq, q, g_mean, g_cov, level_idx=None, noise_idx=None, mean_idx=None,
                              include_noise: bool = False, out=None):
        """d_xq [b*q, dq] = d/d xq of sum(g_mean * mean) + sum(g_cov * cov) of ``posterior_qbatch`` at the same
        arguments (gpp_posterior_qbatch_grad).  ``g_mean`` [b, q] and ``g_cov`` [b, q, q] may be None (zero) and live
        on the host or on this engine's GPU, like the other inputs."""
        xq, m, level_idx, noise_idx, mean_idx = self._candidates(xq, level_idx, noise_idx, mean_idx)
        b, q = self._tbatches(m, q, "posterior_qbatch")
        g = []
        for a, n in ((g_mean, b * q), (g_cov, b * q * q)):
            if a is not None and (isinstance(a, np.ndarray) or not hasattr(a, "data_ptr")):
                a = _f64(a)
            if a is not None and int(np.prod(a.shape)) != n:
                raise ValueError("posterior_qbatch_grad: upstream gradient of %d entries, expected %d"
                                 % (int(np.prod(a.shape)), n))
            g.append(a)
        d_xq = np.empty((b * q, self.dq)) if out is None else out
        rc = self._lib.gpp_posterior_qbatch_grad(self._h, b, q, _ptr(xq), _ptr(level_idx), _ptr(noise_idx),
                                                 _ptr(mean_idx), 1 if include_noise else 0, _ptr(g[0]), _ptr(g[1]),
                                                 _ptr(d_xq))
        if rc != GPP_OK:
            _raise(rc, "gpp_posterior_qbatch_grad")
        return d_xq

    def acquisition_qbatch(self, xq, q_tot, kind, base_samples, best_f: float = 0.0, beta: float = 0.0,
                           n_baseline: int = 0, maximize: bool = True, want_grad: bool = True, level_idx=None,
                           noise_idx=None, mean_idx=None, include_noise: bool = False, out_values=None,
                           out_d_xq=None):
        """Monte-Carlo batch acquisition of the b t-batches of q_tot consecutive rows of ``xq`` (gpp_acq_qbatch):
        returns ``(values [b], d_xq [b*q_tot, dq] or None, jitter [b])`` in scaled y units.  ``kind`` is QACQ_EI,
        QACQ_NEI (the last ``n_baseline`` rows of each t-batch are baseline points) or QACQ_UCB; ``base_samples``
        [S, q_tot] are shared by every t-batch.  ``d_xq`` is d(sum values)/d xq, computed only when ``want_grad``.
        Inputs, base samples and output buffers may live on the host or on this engine's GPU, like ``predict``'s."""
        xq, m, level_idx, noise_idx, mean_idx = self._candidates(xq, level_idx, noise_idx, mean_idx)
        b, q_tot = self._tbatches(m, q_tot, "acquisition_qbatch", "q_tot")
        if isinstance(base_samples, np.ndarray) or not hasattr(base_samples, "data_ptr"):
            base_samples = _f64(base_samples)
        if len(base_samples.shape) != 2 or int(base_samples.shape[1]) != q_tot:
            raise ValueError("acquisition_qbatch: base_samples must have shape [S, %d], got %s"
                             % (q_tot, tuple(base_samples.shape)))
        values = np.empty(b) if out_values is None else out_values
        d_xq = None
        if want_grad:
            d_xq = np.empty((m, self.dq)) if out_d_xq is None else out_d_xq
        jitter = np.empty(b)
        rc = self._lib.gpp_acq_qbatch(self._h, b, q_tot, _ptr(xq), _ptr(level_idx), _ptr(noise_idx), _ptr(mean_idx),
                                      1 if include_noise else 0, int(kind), int(n_baseline), float(best_f),
                                      float(beta), 1 if maximize else 0, int(base_samples.shape[0]),
                                      _ptr(base_samples), _ptr(values), _ptr(d_xq), _ptr(jitter))
        if rc != GPP_OK:
            _raise(rc, "gpp_acq_qbatch")
        return values, d_xq, jitter

    def ipv_points(self, xq, level_idx=None):
        """Stores the integration set of ``nipv_qbatch`` (gpp_ipv_points): the m rows of ``xq`` (and their
        ``level_idx``), host arrays or tensors on this engine's GPU, 1 <= m <= MAX_IPV_POINTS.  The set belongs to the
        current factor: after ``factorize`` or ``mll_grad`` it has to be stored again."""
        xq, m, level_idx, _, _ = self._candidates(xq, level_idx, None, None)
        rc = self._lib.gpp_ipv_points(self._h, m, _ptr(xq), _ptr(level_idx))
        if rc != GPP_OK:
            _raise(rc, "gpp_ipv_points")

    def nipv_qbatch(self, xq, q, want_grad: bool = True, level_idx=None, noise_idx=None, out_values=None,
                    out_d_xq=None):
        """Negative integrated posterior variance over the stored integration set of the b t-batches of q consecutive
        rows of ``xq``, each fantasised with the observation noise of its rows' ``noise_idx`` groups (gpp_nipv_qbatch):
        returns ``(values [b], d_xq [b*q, dq] or None, jitter [b])`` in scaled y units.  ``d_xq`` is
        d(sum values)/d xq, computed only when ``want_grad``.  Inputs and output buffers may live on the host or on
        this engine's GPU, like ``predict``'s."""
        xq, m, level_idx, noise_idx, _ = self._candidates(xq, level_idx, noise_idx, None)
        b, q = self._tbatches(m, q, "nipv_qbatch")
        values = np.empty(b) if out_values is None else out_values
        d_xq = None
        if want_grad:
            d_xq = np.empty((m, self.dq)) if out_d_xq is None else out_d_xq
        jitter = np.empty(b)
        rc = self._lib.gpp_nipv_qbatch(self._h, b, q, _ptr(xq), _ptr(level_idx), _ptr(noise_idx), _ptr(values),
                                       _ptr(d_xq), _ptr(jitter))
        if rc != GPP_OK:
            _raise(rc, "gpp_nipv_qbatch")
        return values, d_xq, jitter

    def kg_qbatch(self, xq, q, n_fantasies, base_samples, maximize: bool = True, want_grad: bool = True,
                  level_idx=None, noise_idx=None, mean_idx=None, out_values=None, out_d_xq=None):
        """One-shot knowledge gradient of the b t-batches of q + n_fantasies consecutive rows of ``xq``, the q actual
        points followed by the fantasy solutions (gpp_kg_qbatch): returns ``(values [b], d_xq [b*q_tot, dq] or None,
        jitter [b])`` in scaled y units.  Each value is the mean over the fantasies f of the posterior mean at fantasy
        solution f after also observing the actual points (with their ``noise_idx`` groups' noise) at their posterior
        mean plus L e_f; ``base_samples`` [n_fantasies, q] are shared by every t-batch.  ``d_xq`` is
        d(sum values)/d xq for all rows, computed only when ``want_grad``.  Inputs, base samples and output buffers
        may live on the host or on this engine's GPU, like ``predict``'s."""
        xq, m, level_idx, noise_idx, mean_idx = self._candidates(xq, level_idx, noise_idx, mean_idx)
        q, nf = int(q), int(n_fantasies)
        if q < 1 or nf < 1:
            raise ValueError("kg_qbatch: q and n_fantasies must be >= 1, got %d and %d" % (q, nf))
        b, q_tot = self._tbatches(m, q + nf, "kg_qbatch", "q + n_fantasies")
        if isinstance(base_samples, np.ndarray) or not hasattr(base_samples, "data_ptr"):
            base_samples = _f64(base_samples)
        if tuple(int(n) for n in base_samples.shape) != (nf, q):
            raise ValueError("kg_qbatch: base_samples must have shape [%d, %d], got %s"
                             % (nf, q, tuple(base_samples.shape)))
        values = np.empty(b) if out_values is None else out_values
        d_xq = None
        if want_grad:
            d_xq = np.empty((m, self.dq)) if out_d_xq is None else out_d_xq
        jitter = np.empty(b)
        rc = self._lib.gpp_kg_qbatch(self._h, b, q, nf, _ptr(xq), _ptr(level_idx), _ptr(noise_idx), _ptr(mean_idx),
                                     1 if maximize else 0, _ptr(base_samples), _ptr(values), _ptr(d_xq),
                                     _ptr(jitter))
        if rc != GPP_OK:
            _raise(rc, "gpp_kg_qbatch")
        return values, d_xq, jitter

    def gibbon_qbatch(self, xq, q, max_values, projected: bool = False, maximize: bool = True,
                      want_grad: bool = True, level_idx=None, noise_idx=None, mean_idx=None, out_values=None,
                      out_d_xq=None):
        """GIBBON values of the b t-batches of q_tot consecutive rows of ``xq`` (gpp_gibbon_qbatch): the q actual points,
        then with ``projected`` their copies at the target fidelity (q_tot = 2q; otherwise q_tot = q).  Returns
        ``(values [b], d_xq [b*q_tot, dq] or None, jitter [b])``, values in nats.  ``max_values`` [K] are samples of
        the maximum of sigma f in scaled y units, shared by every t-batch; the actual rows are observed with their
        ``noise_idx`` groups' noise.  ``d_xq`` is d(sum values)/d xq for all rows, computed only when ``want_grad``.
        Inputs, max values and output buffers may live on the host or on this engine's GPU, like ``predict``'s."""
        xq, m, level_idx, noise_idx, mean_idx = self._candidates(xq, level_idx, noise_idx, mean_idx)
        q = int(q)
        if q < 1:
            raise ValueError("gibbon_qbatch: q must be >= 1, got %d" % q)
        b, q_tot = self._tbatches(m, 2 * q if projected else q, "gibbon_qbatch", "q_tot")
        if isinstance(max_values, np.ndarray) or not hasattr(max_values, "data_ptr"):
            max_values = _f64(max_values).reshape(-1)
        if len(max_values.shape) != 1:
            raise ValueError("gibbon_qbatch: max_values must be one-dimensional, got %s" % (tuple(max_values.shape),))
        values = np.empty(b) if out_values is None else out_values
        d_xq = None
        if want_grad:
            d_xq = np.empty((m, self.dq)) if out_d_xq is None else out_d_xq
        jitter = np.empty(b)
        rc = self._lib.gpp_gibbon_qbatch(self._h, b, q, 1 if projected else 0, _ptr(xq), _ptr(level_idx),
                                         _ptr(noise_idx), _ptr(mean_idx), 1 if maximize else 0,
                                         int(max_values.shape[0]), _ptr(max_values), _ptr(values), _ptr(d_xq),
                                         _ptr(jitter))
        if rc != GPP_OK:
            _raise(rc, "gpp_gibbon_qbatch")
        return values, d_xq, jitter

    def max_value_quartiles(self, xq, level_idx=None, mean_idx=None, maximize: bool = True, out=None):
        """Quartiles [3] (p = 1/4, 1/2, 3/4) of the maximum of sigma f over the m rows of ``xq`` under their
        independent posterior marginals (``predict`` at min_var = 1e-8), in scaled y units
        (gpp_max_value_quartiles).  Inputs and the output buffer may live on the host or on this engine's GPU."""
        xq, m, level_idx, _, mean_idx = self._candidates(xq, level_idx, None, mean_idx)
        quartiles = np.empty(3) if out is None else out
        rc = self._lib.gpp_max_value_quartiles(self._h, m, _ptr(xq), _ptr(level_idx), _ptr(mean_idx),
                                               1 if maximize else 0, _ptr(quartiles))
        if rc != GPP_OK:
            _raise(rc, "gpp_max_value_quartiles")
        return quartiles

    def acq_argmax(self, xq, cost_idx, cost: Sequence[float], kind_by_cost: Sequence[int], best_f: Sequence[float],
                   level_idx=None, mean_idx=None, maximize: bool = True, si: float = 0.0, y_min: float = 0.0,
                   y_std: float = 1.0, min_var: float = 1e-10, return_scores: bool = False):
        host = isinstance(xq, np.ndarray) or not hasattr(xq, "data_ptr")
        if host:
            xq = _f64(xq)
            m = xq.shape[0] if xq.ndim == 2 else (xq.size // max(self.dq, 1))
            level_idx, mean_idx, cost_idx = _i32(level_idx, m), _i32(mean_idx, m), _i32(cost_idx, m)
        else:
            m = int(xq.shape[0])
        cost = _f64(cost).reshape(-1)
        n_cost = cost.shape[0]
        kinds = np.ascontiguousarray(np.asarray(kind_by_cost, dtype=np.int32)).reshape(n_cost)
        bf = _f64(best_f).reshape(n_cost)
        scores = np.empty(m) if return_scores else None
        best = C.c_double()
        idx = C.c_int64()
        rc = self._lib.gpp_acq_argmax(self._h, m, _ptr(xq), _ptr(level_idx), _ptr(mean_idx), _ptr(cost_idx), n_cost,
                                      _ptr(cost), _ptr(kinds), _ptr(bf), 1 if maximize else 0, float(si),
                                      float(y_min), float(y_std), float(min_var), _ptr(scores), C.byref(best),
                                      C.byref(idx))
        if rc != GPP_OK:
            _raise(rc, "gpp_acq_argmax")
        if return_scores:
            return best.value, idx.value, scores
        return best.value, idx.value


def probe_dgemm(m: int, n: int, k: int, iters: int = 10, device: int = 0) -> float:
    """Average milliseconds of one FP64 DMMA GEMM launch C[m,n] = A[m,k] B[n,k]^T."""
    ms = C.c_float()
    rc = load_library().gpp_probe_dgemm(device, m, n, k, iters, C.byref(ms))
    if rc != GPP_OK:
        _raise(rc, "gpp_probe_dgemm")
    return float(ms.value)


FP64_DMMA, FP64_INT8 = 0, 1


def set_fp64_mode(mode: int) -> int:
    """Arithmetic of the O(N^3) stages for engines created afterwards: -1 by size (default), FP64_DMMA, FP64_INT8
    (include/gpplus_b200.h).  Returns the previous setting."""
    return int(load_library().gpp_set_fp64_mode(int(mode)))


def probe_i8(n_cols: int = 256, iters: int = 4096, device: int = 0) -> float:
    """Raw tcgen05 kind::i8 issue rate of the GPU in int8 tera-ops per second (gpp_probe_i8)."""
    tops = C.c_double(0.0)
    rc = load_library().gpp_probe_i8(device, n_cols, iters, C.byref(tops))
    if rc != 0:
        _raise(rc, "gpp_probe_i8")
    return float(tops.value)
