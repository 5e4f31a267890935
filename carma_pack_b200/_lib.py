"""ctypes binding of the C ABI in include/carma_b200.h (libcarma_b200.so).

This is the only way Python reaches the GPU path.  There is no CPU fallback: if the shared
library is missing the import fails loudly, and every compute call raises CarmaError when CUDA is
unavailable.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CARMA_B200_LIB") or os.path.join(_HERE, "libcarma_b200.so")  # override: tuning builds


def _point_at_bundled_nccl():
    """The library loads NCCL lazily (carma_comm_* / carma_gather_summaries).  When this Python environment ships a
    pip-bundled NCCL (the one torch links against), make that the copy that gets mapped, so that a later
    `import torch` in the same process finds the symbols it needs behind the soname libnccl.so.2.  torch itself is not
    imported here."""
    if os.environ.get("CARMA_NCCL_LIB"):
        return
    try:
        import importlib.util
        spec = importlib.util.find_spec("nvidia.nccl")
        for loc in (spec.submodule_search_locations if spec else []):
            cand = os.path.join(loc, "lib", "libnccl.so.2")
            if os.path.exists(cand):
                os.environ["CARMA_NCCL_LIB"] = cand
                return
    except Exception:  # noqa: BLE001 - best effort: the system NCCL is the fallback
        pass


_point_at_bundled_nccl()

KIND_CAR1, KIND_CARP, KIND_CARMA, KIND_ZCAR, KIND_ZCARMA = 0, 1, 2, 3, 4
IGNORE_BOUNDS, LOGLIK_ONLY = 1, 2
MAX_P = 7
# status of MultiSeries.hessian per curve (CARMA_HESS_*), and its default relative step 2^-13
HESS_OK, HESS_REJECTED, HESS_NONFINITE, HESS_NOT_NEGDEF = 0, 1, 2, 3
HESS_REL_STEP = 2.0 ** -13
# status of MultiSeries.laplace per curve (CARMA_LAPLACE_*), and the most draws per curve of one call
LAPLACE_OK, LAPLACE_BAD_COV, LAPLACE_NO_WEIGHT = 0, 1, 2
LAPLACE_MAX_DRAWS = 1 << 20

EXPORTED_SYMBOLS = [
    "carma_last_error", "carma_abi_version", "carma_device_count",
    "carma_series_create", "carma_series_destroy", "carma_series_length", "carma_series_default_prior",
    "carma_loglik_batch_dev", "carma_loglik_batch", "carma_loglik_batch_async", "carma_loglik_batch_wait",
    "carma_log_prior", "carma_loglik_scan_dev", "carma_loglik_scan",
    "carma_multi_series_create", "carma_multi_series_destroy", "carma_multi_series_default_priors",
    "carma_multi_series_simulate", "carma_multi_series_get_curve",
    "carma_mle_default_opts", "carma_mle_batch", "carma_lbfgs_batch",
    "carma_multi_loglik_dev", "carma_multi_loglik",
    "carma_filter", "carma_predict",
    "carma_pt_default_opts", "carma_pt_run", "carma_pt_run_dev", "carma_multi_pt_run",
    "carma_fp64_peak_tflops", "carma_philox_dev", "carma_tdist_dev", "carma_fastmath_dev",
    "carma_simulate", "carma_starting_value", "carma_comm_unique_id", "carma_comm_init_rank", "carma_comm_destroy",
    "carma_gather_summaries", "carma_gather_summaries_dev", "carma_derived_params", "carma_derived_params_dev", "carma_mle_batch_device",
    "carma_mle_grid_device", "carma_multi_series_curve_stats", "carma_multi_mle_grid_device",
    "carma_multi_filter_dev", "carma_multi_filter", "carma_multi_assess_fit", "carma_multi_predict",
    "carma_multi_simulate", "carma_psd_quantiles", "carma_psd_quantiles_dev", "carma_effective_samples",
    "carma_effective_samples_dev", "carma_multi_smooth", "carma_multi_hessian", "carma_multi_laplace",
]


class CarmaError(RuntimeError):
    pass


class Prior(ctypes.Structure):
    _fields_ = [("max_stdev", ctypes.c_double), ("max_freq", ctypes.c_double), ("min_freq", ctypes.c_double),
                ("kappa_low", ctypes.c_double), ("kappa_high", ctypes.c_double), ("measerr_dof", ctypes.c_double)]

    def as_tuple(self):
        return (self.max_stdev, self.max_freq, self.min_freq, self.kappa_low, self.kappa_high, self.measerr_dof)


PRIOR_DTYPE = np.dtype([("max_stdev", "f8"), ("max_freq", "f8"), ("min_freq", "f8"), ("kappa_low", "f8"),
                        ("kappa_high", "f8"), ("measerr_dof", "f8")])


class PTOpts(ctypes.Structure):
    _fields_ = [("nsamples", ctypes.c_int), ("burnin", ctypes.c_int), ("thin", ctypes.c_int),
                ("ntemps", ctypes.c_int), ("tmax", ctypes.c_double), ("dof", ctypes.c_int),
                ("target_rate", ctypes.c_double), ("gamma", ctypes.c_double), ("seed", ctypes.c_uint64),
                ("ensemble_offset", ctypes.c_uint32), ("max_start_attempts", ctypes.c_int),
                ("order_mode", ctypes.c_int), ("record_trace", ctypes.c_int)]


class MLEJob(ctypes.Structure):   # carma_mle_job_t
    _fields_ = [("kind", ctypes.c_int), ("p", ctypes.c_int), ("q", ctypes.c_int), ("flags", ctypes.c_uint),
                ("prior", Prior), ("nstart", ctypes.c_size_t)]


MAX_DIM = 17   # CARMA_MAX_DIM


class CurveStats(ctypes.Structure):   # carma_curve_stats_t
    _fields_ = [("y_mean", ctypes.c_double), ("y_var_pop", ctypes.c_double), ("y_var_sample", ctypes.c_double),
                ("min_dt", ctypes.c_double), ("median_dt", ctypes.c_double), ("tspan", ctypes.c_double),
                ("dt_max", ctypes.c_double), ("ny", ctypes.c_int64)]


CURVE_STATS_DTYPE = np.dtype([(name, "f8" if ct is ctypes.c_double else "i8") for name, ct in CurveStats._fields_])


class MLEOpts(ctypes.Structure):
    _fields_ = [("maxiter", ctypes.c_int), ("history", ctypes.c_int), ("max_backtrack", ctypes.c_int),
                ("reserved", ctypes.c_int), ("gtol", ctypes.c_double), ("ftol", ctypes.c_double),
                ("fd_eps", ctypes.c_double)]


TRACE_DTYPE = np.dtype([("lp_prop", "f8"), ("lp_cur", "f8"), ("alpha", "f8"), ("u", "f8"),
                        ("accepted", "i4"), ("pad", "i4")])

_dp = ctypes.POINTER(ctypes.c_double)
_vp = ctypes.c_void_p
_sz = ctypes.c_size_t
OBJECTIVE_FN = ctypes.CFUNCTYPE(ctypes.c_int, _dp, _sz, _sz, _dp, _vp)


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "carma_pack_b200: %s is missing. Build it with `python build_native.py` "
            "(nvcc, sm_100a). There is no CPU fallback." % LIB_PATH)
    L = ctypes.CDLL(LIB_PATH)
    L.carma_last_error.restype = ctypes.c_char_p
    pr = ctypes.POINTER(Prior)
    L.carma_series_create.argtypes = [_dp, _dp, _dp, _sz, ctypes.c_int, ctypes.POINTER(_vp)]
    L.carma_series_destroy.argtypes = [_vp]
    L.carma_series_length.argtypes = [_vp, ctypes.POINTER(_sz)]
    L.carma_series_default_prior.argtypes = [_vp, ctypes.c_int, pr]
    L.carma_loglik_batch_dev.argtypes = [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, pr, _sz, _vp, _vp,
                                         ctypes.c_uint, _vp]
    L.carma_loglik_batch.argtypes = [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, pr, _sz, _vp, _vp, ctypes.c_uint]
    L.carma_loglik_scan_dev.argtypes = [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, pr, _sz, _vp, _vp,
                                        ctypes.c_uint, ctypes.c_int, _vp]
    L.carma_loglik_scan.argtypes = [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, pr, _sz, _vp, _vp, ctypes.c_uint,
                                    ctypes.c_int]
    L.carma_loglik_batch_async.argtypes = [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, pr, _sz, _vp, _vp,
                                           ctypes.c_uint, ctypes.c_int]
    L.carma_loglik_batch_wait.argtypes = [_vp, ctypes.c_int]
    L.carma_log_prior.argtypes = [ctypes.c_int, ctypes.c_int, _dp, pr, _dp]
    L.carma_multi_series_create.argtypes = [_dp, _dp, _dp, ctypes.POINTER(ctypes.c_int64), _sz, ctypes.c_int,
                                            ctypes.POINTER(_vp)]
    L.carma_multi_series_destroy.argtypes = [_vp]
    L.carma_multi_series_default_priors.argtypes = [_vp, ctypes.c_int, _vp]
    L.carma_multi_series_simulate.argtypes = [_sz, _sz, ctypes.c_int, ctypes.c_int, ctypes.c_int, _dp, pr,
                                              ctypes.c_double, ctypes.c_double, ctypes.c_double, ctypes.c_uint64,
                                              ctypes.c_uint32, ctypes.c_int, ctypes.POINTER(_vp)]
    L.carma_multi_series_get_curve.argtypes = [_vp, _sz, _dp, _dp, _dp, _sz, ctypes.POINTER(_sz)]
    L.carma_mle_default_opts.argtypes = [ctypes.POINTER(MLEOpts)]
    L.carma_mle_default_opts.restype = None
    L.carma_lbfgs_batch.argtypes = [OBJECTIVE_FN, _vp, _sz, _sz, _dp, _dp, _dp, ctypes.POINTER(MLEOpts), _dp, _dp,
                                    ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_longlong)]
    L.carma_mle_batch.argtypes = [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, pr, ctypes.c_uint, _sz, _dp, _dp, _dp,
                                  ctypes.POINTER(MLEOpts), _dp, _dp, ctypes.POINTER(ctypes.c_int),
                                  ctypes.POINTER(ctypes.c_longlong), ctypes.c_int]
    L.carma_mle_batch_device.argtypes = L.carma_mle_batch.argtypes
    L.carma_mle_grid_device.argtypes = [_vp, ctypes.c_int, ctypes.POINTER(MLEJob), _dp, _dp, _dp, ctypes.POINTER(MLEOpts),
                                        _dp, _dp, ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_longlong), ctypes.c_int]
    L.carma_multi_series_curve_stats.argtypes = [_vp, _vp]
    L.carma_multi_mle_grid_device.argtypes = [_vp, ctypes.c_int, ctypes.POINTER(MLEJob), _vp, _dp, _dp, _dp,
                                              ctypes.POINTER(MLEOpts), _dp, _dp, ctypes.POINTER(ctypes.c_int),
                                              ctypes.POINTER(ctypes.c_longlong)]
    L.carma_multi_loglik_dev.argtypes = [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, _vp, _vp, _vp,
                                         ctypes.c_uint, _vp]
    L.carma_multi_loglik.argtypes = [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, _vp, _vp, _vp, ctypes.c_uint]
    L.carma_multi_filter_dev.argtypes = [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, _vp, _vp, ctypes.c_uint, _vp, _vp,
                                         _vp, _vp]
    L.carma_multi_filter.argtypes = [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, _vp, _vp, ctypes.c_uint, _vp, _vp, _vp]
    L.carma_multi_assess_fit.argtypes = [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, _vp, _vp, ctypes.c_uint,
                                         ctypes.c_int, _vp]
    L.carma_multi_predict.argtypes = [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, _vp, _vp, ctypes.c_uint, _vp, _vp,
                                      _vp, _vp]
    L.carma_multi_simulate.argtypes = [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, _vp, _vp, _sz, ctypes.c_uint, _vp,
                                       _vp, _sz, ctypes.c_uint64, ctypes.c_uint32, _vp]
    L.carma_multi_smooth.argtypes = [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, _vp, _vp, ctypes.c_uint, _vp, _vp, _vp,
                                     _vp, _vp, _vp, _vp, _vp, _vp]
    L.carma_multi_hessian.argtypes = [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, _vp, _vp, ctypes.c_uint,
                                      ctypes.c_double, _vp, _vp, _vp, _vp, _vp]
    L.carma_multi_laplace.argtypes = [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, _vp, _vp, _vp, ctypes.c_uint, _sz,
                                      ctypes.c_uint64, ctypes.c_uint32, _vp, _vp, _vp, _vp, _vp, _vp, _vp]
    L.carma_filter.argtypes = [_vp, ctypes.c_double, _dp, _dp, ctypes.c_int, ctypes.c_double, ctypes.c_double, _dp, _dp]
    L.carma_predict.argtypes = [_vp, ctypes.c_double, _dp, _dp, ctypes.c_int, ctypes.c_double, ctypes.c_double,
                                _dp, _sz, _dp, _dp]
    L.carma_pt_default_opts.argtypes = [ctypes.POINTER(PTOpts)]
    L.carma_pt_default_opts.restype = None
    L.carma_pt_run.argtypes = [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, pr, ctypes.POINTER(PTOpts), _sz,
                               _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]
    L.carma_pt_run_dev.argtypes = [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, pr, ctypes.POINTER(PTOpts), _sz,
                                   _vp, _vp, _vp, _vp, _vp, _vp]
    L.carma_multi_pt_run.argtypes = [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, _vp, ctypes.POINTER(PTOpts), _sz,
                                     _vp, _vp, _vp, _vp]
    L.carma_fp64_peak_tflops.argtypes = [ctypes.c_int, _dp]
    L.carma_philox_dev.argtypes = [ctypes.c_uint32] * 4 + [ctypes.c_uint64, ctypes.POINTER(ctypes.c_uint32)]
    L.carma_fastmath_dev.argtypes = [_dp, _dp, _sz, _dp, _dp, _dp, _dp, _dp, _dp]
    L.carma_simulate.argtypes = [_vp, ctypes.c_double, _dp, _dp, ctypes.c_int, ctypes.c_double, ctypes.c_double, _dp, _sz,
                                 ctypes.c_uint64, _sz, _dp]
    L.carma_starting_value.argtypes = [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.POINTER(Prior), ctypes.c_uint64,
                                       ctypes.c_uint32, ctypes.c_int, _dp, _dp]
    L.carma_derived_params.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, _sz, _dp, _dp, ctypes.c_int]
    L.carma_derived_params_dev.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, _sz, _vp, _vp, _vp]
    L.carma_psd_quantiles.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, _vp, _sz, _sz, _vp, _vp, _sz, _sz, _vp, _sz,
                                      _vp, _vp, ctypes.c_int]
    L.carma_psd_quantiles_dev.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, _vp, _sz, _sz, _vp, _vp, _sz, _sz, _vp,
                                          _sz, _vp, _vp, _vp]
    L.carma_effective_samples.argtypes = [_sz, _sz, _sz, _vp, _vp, ctypes.c_int]
    L.carma_effective_samples_dev.argtypes = [_sz, _sz, _sz, _vp, _vp, _vp]
    L.carma_comm_unique_id.argtypes = [ctypes.c_char_p]
    L.carma_comm_init_rank.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_char_p, ctypes.c_int, ctypes.POINTER(ctypes.c_void_p)]
    L.carma_comm_destroy.argtypes = [_vp]
    L.carma_gather_summaries.argtypes = [_vp, _dp, _sz, _dp, _vp]
    L.carma_gather_summaries_dev.argtypes = [_vp, _vp, _sz, _vp, _vp]
    L.carma_tdist_dev.argtypes = [ctypes.c_uint64, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_int, _dp]
    return L


lib = _load()


def check(rc, what=""):
    if rc != 0:
        msg = lib.carma_last_error()
        raise CarmaError("%s failed (code %d): %s" % (what, rc, msg.decode() if msg else ""))


def model_dim(kind, p, q):
    if kind == KIND_CAR1:
        return 4
    if kind == KIND_CARMA:
        return 3 + p + q
    if kind == KIND_ZCARMA:
        return 4 + p
    return 3 + p


def _c(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _ptr(a):
    return a.ctypes.data_as(_dp)


def device_count():
    n = ctypes.c_int(0)
    rc = lib.carma_device_count(ctypes.byref(n))
    return n.value if rc == 0 else 0


def derived_params(kind, p, q, theta, prior=None, device=0):
    """Posterior post-processing on the device (carma_derived_params): theta rows -> dict of ar_roots (complex, n x p),
    ar_coefs (n x p+1, highest power first), ma_coefs (n x p, beta_0 = 1, zero beyond q), sigma (n), psd_width and
    psd_centroid (n x p)."""
    th = np.ascontiguousarray(np.atleast_2d(theta), dtype=np.float64)
    d = model_dim(kind, p, q)
    if th.shape[1] != d:
        raise ValueError("theta must have %d columns for this model, got %d" % (d, th.shape[1]))
    n = th.shape[0]
    out = np.empty((n, 6 * p + 2))
    check(lib.carma_derived_params(kind, p, q, ctypes.byref(prior) if prior is not None else None, n, _ptr(th), _ptr(out),
                                   device), "carma_derived_params")
    return {"ar_roots": out[:, 0:2 * p:2] + 1j * out[:, 1:2 * p:2], "ar_coefs": out[:, 2 * p:3 * p + 1].copy(),
            "ma_coefs": out[:, 3 * p + 1:4 * p + 1].copy(), "sigma": out[:, 4 * p + 1].copy(),
            "psd_width": out[:, 4 * p + 2:5 * p + 2].copy(), "psd_centroid": out[:, 5 * p + 2:6 * p + 2].copy()}


def psd_quantiles(kind, p, q, theta, freq, percentiles, priors=None, return_psd=False, device=0):
    """Pointwise percentiles of the power spectrum over each curve's samples (carma_psd_quantiles).  theta (ncurves,
    nsamples, d); freq (nfreq,) shared by every curve or (ncurves, nfreq); percentiles in [0, 100]; priors: ncurves
    entries of PRIOR_DTYPE (only the kappa bounds are read; required for ZCARMA).  Returns out (ncurves, npct, nfreq),
    bitwise np.percentile(psd, percentiles, axis=1) of the kernel's PSD values, and with return_psd=True also those
    values, psd (ncurves, nsamples, nfreq)."""
    th = np.ascontiguousarray(theta, dtype=np.float64)
    d = model_dim(kind, p, q)
    if th.ndim != 3 or th.shape[2] != d:
        raise ValueError("theta must be (ncurves, nsamples, %d)" % d)
    nc, ns = th.shape[0], th.shape[1]
    fr = _c(freq)
    if fr.ndim == 1:
        rows = 1
    elif fr.ndim == 2 and fr.shape[0] == nc:
        rows = nc
    else:
        raise ValueError("freq must be (nfreq,) or (%d, nfreq)" % nc)
    nf = fr.shape[-1]
    pct = _c(np.atleast_1d(percentiles))
    if pct.ndim != 1:
        raise ValueError("percentiles must be a scalar or a 1-d sequence")
    pp = None
    if priors is not None:
        priors = np.ascontiguousarray(priors, dtype=PRIOR_DTYPE)
        if priors.shape != (nc,):
            raise ValueError("priors must have %d entries" % nc)
        pp = priors.ctypes.data
    out = np.empty((nc, pct.size, nf))
    psd = np.empty((nc, ns, nf)) if return_psd else None
    check(lib.carma_psd_quantiles(kind, p, q, pp, nc, ns, th.ctypes.data, fr.ctypes.data, rows, nf, pct.ctypes.data,
                                  pct.size, out.ctypes.data, psd.ctypes.data if return_psd else None, device),
          "carma_psd_quantiles")
    return (out, psd) if return_psd else out


def effective_samples(x, device=0):
    """MCMCSample.effective_samples for every column of every series (carma_effective_samples): x (nseries, n, k) ->
    ess (nseries, k)."""
    xs = np.ascontiguousarray(x, dtype=np.float64)
    if xs.ndim != 3:
        raise ValueError("x must be (nseries, n, k)")
    ns, n, k = xs.shape
    ess = np.empty((ns, k))
    check(lib.carma_effective_samples(ns, n, k, xs.ctypes.data, ess.ctypes.data, device), "carma_effective_samples")
    return ess


class Series:
    """One light curve resident in HBM (carma_series_t)."""

    def __init__(self, time, y, yerr, device=0):
        t, yy, ee = _c(time), _c(y), _c(yerr)
        if not (t.shape == yy.shape == ee.shape and t.ndim == 1):
            raise ValueError("time, y, yerr must be 1-d arrays of equal length")
        self.handle = _vp()
        check(lib.carma_series_create(_ptr(t), _ptr(yy), _ptr(ee), t.size, device, ctypes.byref(self.handle)),
              "carma_series_create")
        self.ny = t.size
        self.device = device
        self.time, self.y, self.yerr = t, yy, ee

    def close(self):
        if getattr(self, "handle", None):
            lib.carma_series_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def default_prior(self, population_var=True):
        pr = Prior()
        check(lib.carma_series_default_prior(self.handle, int(population_var), ctypes.byref(pr)), "default_prior")
        return pr

    def loglik(self, kind, p, q, theta, prior=None, flags=0):
        """Batched CARMA_Base::LogDensity with host arrays (H2D + kernel + D2H inside)."""
        th = np.ascontiguousarray(np.atleast_2d(theta), dtype=np.float64)
        d = model_dim(kind, p, q)
        if th.shape[1] != d:
            raise ValueError("theta must have %d columns for this model, got %d" % (d, th.shape[1]))
        if prior is None:
            prior = self.default_prior()
        out = np.empty(th.shape[0])
        check(lib.carma_loglik_batch(self.handle, kind, p, q, ctypes.byref(prior), th.shape[0],
                                     th.ctypes.data, out.ctypes.data, flags), "carma_loglik_batch")
        return out

    def loglik_async(self, kind, p, q, theta_ptr, out_ptr, n, prior, slot, flags=0):
        """Enqueue H2D + kernel + D2H for host buffers (raw addresses, ideally pinned) on pipeline slot 0/1."""
        check(lib.carma_loglik_batch_async(self.handle, kind, p, q, ctypes.byref(prior), n, theta_ptr, out_ptr, flags,
                                           slot), "carma_loglik_batch_async")

    def loglik_wait(self, slot):
        check(lib.carma_loglik_batch_wait(self.handle, slot), "carma_loglik_batch_wait")

    def loglik_scan(self, kind, p, q, theta, prior=None, flags=0, chunk=0):
        """Same value as loglik(), computed by the temporally parallel scan (for one very long series)."""
        th = np.ascontiguousarray(np.atleast_2d(theta), dtype=np.float64)
        d = model_dim(kind, p, q)
        if th.shape[1] != d:
            raise ValueError("theta must have %d columns for this model, got %d" % (d, th.shape[1]))
        if prior is None:
            prior = self.default_prior()
        out = np.empty(th.shape[0])
        check(lib.carma_loglik_scan(self.handle, kind, p, q, ctypes.byref(prior), th.shape[0], th.ctypes.data,
                                    out.ctypes.data, flags, chunk), "carma_loglik_scan")
        return out

    def loglik_scan_dev(self, kind, p, q, d_theta_ptr, d_out_ptr, n, prior, flags=0, chunk=0, stream=0):
        check(lib.carma_loglik_scan_dev(self.handle, kind, p, q, ctypes.byref(prior), n, d_theta_ptr, d_out_ptr, flags,
                                        chunk, stream), "carma_loglik_scan_dev")

    def loglik_dev(self, kind, p, q, d_theta_ptr, d_out_ptr, n, prior, flags=0, stream=0):
        """Device-resident variant: raw device pointers (e.g. torch tensor .data_ptr()), no sync."""
        check(lib.carma_loglik_batch_dev(self.handle, kind, p, q, ctypes.byref(prior), n, d_theta_ptr, d_out_ptr,
                                         flags, stream), "carma_loglik_batch_dev")

    def filter(self, sigsqr, omega, ma, measerr_scale=1.0, mu=0.0):
        om = np.asarray(omega, dtype=complex).ravel()
        p = om.size
        buf = np.empty(2 * p)
        buf[0::2], buf[1::2] = om.real, om.imag
        m = np.zeros(p)
        m[:len(ma)] = ma
        mean, var = np.empty(self.ny), np.empty(self.ny)
        check(lib.carma_filter(self.handle, sigsqr, _ptr(buf), _ptr(m), p, measerr_scale, mu, _ptr(mean), _ptr(var)),
              "carma_filter")
        return mean, var

    def predict(self, sigsqr, omega, ma, tq, measerr_scale=1.0, mu=0.0):
        om = np.asarray(omega, dtype=complex).ravel()
        p = om.size
        buf = np.empty(2 * p)
        buf[0::2], buf[1::2] = om.real, om.imag
        m = np.zeros(p)
        m[:len(ma)] = ma
        q = _c(np.atleast_1d(tq))
        qm, qv = np.empty(q.size), np.empty(q.size)
        check(lib.carma_predict(self.handle, sigsqr, _ptr(buf), _ptr(m), p, measerr_scale, mu, _ptr(q), q.size,
                                _ptr(qm), _ptr(qv)), "carma_predict")
        return qm, qv

    def simulate(self, sigsqr, omega, ma, tsim, measerr_scale=1.0, mu=0.0, seed=1, npaths=1):
        """Conditional simulation of the process at `tsim` given the data (carma_simulate): (npaths, nsim) array."""
        om = np.asarray(omega, dtype=complex).ravel()
        p = om.size
        buf = np.empty(2 * p)
        buf[0::2], buf[1::2] = om.real, om.imag
        m = np.zeros(p)
        m[:len(ma)] = ma
        q = _c(np.atleast_1d(tsim))
        out = np.empty((int(npaths), q.size))
        check(lib.carma_simulate(self.handle, sigsqr, _ptr(buf), _ptr(m), p, measerr_scale, mu, _ptr(q), q.size,
                                 int(seed), int(npaths), _ptr(out)), "carma_simulate")
        return out

    def pt_run(self, kind, p, q, nsamples, burnin, thin=1, ntemps=10, n_ensembles=1, seed=1, ensemble_offset=0,
               init=None, prior=None, order_mode=0, record_trace=False, tmax=100.0, dof=8, target_rate=0.25,
               gamma=2.0 / 3.0, max_start_attempts=1000):
        """RunCarmaSampler for n_ensembles independent ensembles, fully on device."""
        d = model_dim(kind, p, q)
        if prior is None:
            prior = self.default_prior()
        o = PTOpts()
        lib.carma_pt_default_opts(ctypes.byref(o))
        o.nsamples, o.burnin, o.thin, o.ntemps = int(nsamples), int(burnin), int(thin), int(ntemps)
        o.tmax, o.dof, o.target_rate, o.gamma = tmax, dof, target_rate, gamma
        o.seed, o.ensemble_offset, o.max_start_attempts = seed, ensemble_offset, max_start_attempts
        o.order_mode, o.record_trace = order_mode, int(record_trace)
        samples = np.empty((n_ensembles, nsamples, d))
        logposts = np.empty((n_ensembles, nsamples))
        acc = np.empty((n_ensembles, ntemps))
        xr = np.empty((n_ensembles, ntemps))
        iters = burnin + nsamples * thin
        rt = xt = prop = None
        if record_trace:
            rt = np.zeros((n_ensembles, iters, ntemps), dtype=TRACE_DTYPE)
            xt = np.zeros((n_ensembles, iters, ntemps), dtype=TRACE_DTYPE)
            prop = np.zeros((n_ensembles, iters, ntemps, d))
        initp = None
        if init is not None and len(init) == d:
            init = _c(init)
            initp = init.ctypes.data
        check(lib.carma_pt_run(self.handle, kind, p, q, ctypes.byref(prior), ctypes.byref(o), n_ensembles, initp,
                               samples.ctypes.data, logposts.ctypes.data, acc.ctypes.data, xr.ctypes.data,
                               rt.ctypes.data if record_trace else None, xt.ctypes.data if record_trace else None,
                               prop.ctypes.data if record_trace else None), "carma_pt_run")
        res = dict(samples=samples, logposts=logposts, accept_rates=acc, exchange_rates=xr)
        if record_trace:
            res.update(ram_trace=rt, exchange_trace=xt, proposals=prop)
        return res

    def mle_batch(self, kind, p, q, x0, lower, upper, prior=None, flags=0, maxiter=1000, history=8, gtol=1e-5,
                  ftol=2.2e-9, fd_eps=1e-8, slot=0, on_device=False):
        """Projected L-BFGS from every row of x0: minimises -LogDensity over the box [lower, upper].  on_device=False:
        carma_mle_batch (host loop, all rows in lock-step, one launch per batch of trial points); on_device=True:
        carma_mle_batch_device (the whole fit of a start inside one kernel, one warp per start).  Returns
        (x, f, nit, nfev).  Releases the GIL for the whole fit."""
        d = model_dim(kind, p, q)
        x0 = np.ascontiguousarray(x0, dtype=np.float64)
        if x0.ndim != 2 or x0.shape[1] != d:
            raise ValueError("x0 must be (nstart, %d)" % d)
        lo, hi = _c(np.broadcast_to(lower, (d,))), _c(np.broadcast_to(upper, (d,)))
        if prior is None:
            prior = self.default_prior()
        o = MLEOpts()
        lib.carma_mle_default_opts(ctypes.byref(o))
        o.maxiter, o.history, o.gtol, o.ftol, o.fd_eps = int(maxiter), int(history), gtol, ftol, fd_eps
        n = x0.shape[0]
        x, f = np.empty((n, d)), np.empty(n)
        nit, nfev = ctypes.c_int(0), ctypes.c_longlong(0)
        fn = lib.carma_mle_batch_device if on_device else lib.carma_mle_batch
        check(fn(self.handle, kind, p, q, ctypes.byref(prior), flags, n, _ptr(x0), _ptr(lo), _ptr(hi),
                 ctypes.byref(o), _ptr(x), _ptr(f), ctypes.byref(nit), ctypes.byref(nfev), slot),
              "carma_mle_batch_device" if on_device else "carma_mle_batch")
        return x, f, nit.value, nfev.value

    def mle_grid(self, jobs, maxiter=1000, history=8, gtol=1e-5, ftol=2.2e-9, fd_eps=1e-8, slot=0):
        """Several models fitted in one launch (carma_mle_grid_device).  jobs: sequence of (kind, p, q, x0, lower, upper,
        prior, flags), the last six as CarmaModel.mle_starts returns them.  Returns a list of (x, f, nit, nfev), one per job."""
        nj = len(jobs)
        cj = (MLEJob * max(nj, 1))()
        lo = np.zeros((max(nj, 1), MAX_DIM))
        hi = np.zeros((max(nj, 1), MAX_DIM))
        xs, dims = [], []
        for j, (kind, p, q, x0, lower, upper, prior, flags) in enumerate(jobs):
            d = model_dim(kind, p, q)
            x0 = np.ascontiguousarray(x0, dtype=np.float64)
            if x0.ndim != 2 or x0.shape[1] != d:
                raise ValueError("x0 of job %d must be (nstart, %d)" % (j, d))
            lo[j, :d] = np.asarray(lower, dtype=np.float64).reshape(d)
            hi[j, :d] = np.asarray(upper, dtype=np.float64).reshape(d)
            cj[j].kind, cj[j].p, cj[j].q, cj[j].flags, cj[j].nstart = kind, p, q, flags, x0.shape[0]
            cj[j].prior = self.default_prior() if prior is None else prior
            xs.append(x0.reshape(-1))
            dims.append((x0.shape[0], d))
        xin = np.ascontiguousarray(np.concatenate(xs)) if xs else np.zeros(0)
        xout = np.empty_like(xin)
        fout = np.empty(sum(n for n, _ in dims))
        nit = (ctypes.c_int * max(nj, 1))()
        nfev = (ctypes.c_longlong * max(nj, 1))()
        o = MLEOpts()
        lib.carma_mle_default_opts(ctypes.byref(o))
        o.maxiter, o.history, o.gtol, o.ftol, o.fd_eps = maxiter, history, gtol, ftol, fd_eps
        check(lib.carma_mle_grid_device(self.handle, nj, cj, _ptr(xin), _ptr(lo), _ptr(hi), ctypes.byref(o), _ptr(xout),
                                        _ptr(fout), nit, nfev, slot), "carma_mle_grid_device")
        res, ox, of = [], 0, 0
        for j, (n, d) in enumerate(dims):
            res.append((xout[ox:ox + n * d].reshape(n, d).copy(), fout[of:of + n].copy(), int(nit[j]), int(nfev[j])))
            ox += n * d
            of += n
        return res

    def pt_run_dev(self, kind, p, q, opts, n_ensembles, d_samples, d_logposts, prior, d_init=None, d_accept=None,
                   d_exchange=None, stream=0):
        check(lib.carma_pt_run_dev(self.handle, kind, p, q, ctypes.byref(prior), ctypes.byref(opts), n_ensembles,
                                   d_init, d_samples, d_logposts, d_accept, d_exchange, stream), "carma_pt_run_dev")


class MultiSeries:
    """Ragged batch of light curves (CSR offsets) resident in HBM (carma_multi_series_t)."""

    def __init__(self, time, y, yerr, offsets, device=0):
        t, yy, ee = _c(time), _c(y), _c(yerr)
        off = np.ascontiguousarray(offsets, dtype=np.int64)
        self.ncurves = off.size - 1
        self.handle = _vp()
        check(lib.carma_multi_series_create(_ptr(t), _ptr(yy), _ptr(ee),
                                            off.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), self.ncurves, device,
                                            ctypes.byref(self.handle)), "carma_multi_series_create")
        self.offsets = off
        self.device = device

    @classmethod
    def simulate(cls, ncurves, ny, kind, p, q, theta_true, yerr=0.05, dt_min=0.05, dt_max=50.0, seed=0,
                 curve_offset=0, prior=None, device=0):
        """ncurves synthetic light curves of ny points generated in HBM from the model theta_true
        (carma_multi_series_simulate); nothing crosses PCIe except the per-curve statistics."""
        th = _c(theta_true)
        if th.shape != (model_dim(kind, p, q),):
            raise ValueError("theta_true must have %d entries" % model_dim(kind, p, q))
        self = cls.__new__(cls)
        self.ncurves = int(ncurves)
        self.handle = _vp()
        pp = ctypes.byref(prior) if prior is not None else None
        check(lib.carma_multi_series_simulate(int(ncurves), int(ny), kind, p, q, _ptr(th), pp, float(yerr),
                                              float(dt_min), float(dt_max), int(seed), int(curve_offset), device,
                                              ctypes.byref(self.handle)), "carma_multi_series_simulate")
        self.offsets = np.arange(self.ncurves + 1, dtype=np.int64) * int(ny)
        self.device = device
        return self

    def curve(self, c):
        """(time, y, yerr) of curve c copied back to the host; time starts at 0."""
        n = int(self.offsets[c + 1] - self.offsets[c])
        t, y, e = np.empty(n), np.empty(n), np.empty(n)
        got = _sz(0)
        check(lib.carma_multi_series_get_curve(self.handle, int(c), _ptr(t), _ptr(y), _ptr(e), n, ctypes.byref(got)),
              "carma_multi_series_get_curve")
        return t, y, e

    def close(self):
        if getattr(self, "handle", None):
            lib.carma_multi_series_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def default_priors(self, population_var=True):
        out = np.empty(self.ncurves, dtype=PRIOR_DTYPE)
        check(lib.carma_multi_series_default_priors(self.handle, int(population_var), out.ctypes.data), "default_priors")
        return out

    def loglik(self, kind, p, q, theta, priors=None, flags=0):
        th = np.ascontiguousarray(theta, dtype=np.float64)
        d = model_dim(kind, p, q)
        if th.shape != (self.ncurves, d):
            raise ValueError("theta must be (%d, %d)" % (self.ncurves, d))
        out = np.empty(self.ncurves)
        pp = None
        if priors is not None:
            priors = np.ascontiguousarray(priors, dtype=PRIOR_DTYPE)
            pp = priors.ctypes.data
        check(lib.carma_multi_loglik(self.handle, kind, p, q, pp, th.ctypes.data, out.ctypes.data, flags),
              "carma_multi_loglik")
        return out

    def pt_run(self, kind, p, q, nsamples, burnin, thin=1, ntemps=10, n_ensembles=1, seed=1, ensemble_offset=0,
               priors=None, order_mode=0):
        """One PT-MCMC run per light curve (n_ensembles ensembles each), all curves in one launch."""
        d = model_dim(kind, p, q)
        o = PTOpts()
        lib.carma_pt_default_opts(ctypes.byref(o))
        o.nsamples, o.burnin, o.thin, o.ntemps = int(nsamples), int(burnin), int(thin), int(ntemps)
        o.seed, o.ensemble_offset, o.order_mode = seed, ensemble_offset, order_mode
        nc = self.ncurves
        samples = np.empty((nc, n_ensembles, nsamples, d))
        logposts = np.empty((nc, n_ensembles, nsamples))
        acc = np.empty((nc, n_ensembles, ntemps))
        xr = np.empty((nc, n_ensembles, ntemps))
        pp = None
        if priors is not None:
            priors = np.ascontiguousarray(priors, dtype=PRIOR_DTYPE)
            pp = priors.ctypes.data
        check(lib.carma_multi_pt_run(self.handle, kind, p, q, pp, ctypes.byref(o), n_ensembles, samples.ctypes.data,
                                     logposts.ctypes.data, acc.ctypes.data, xr.ctypes.data), "carma_multi_pt_run")
        return dict(samples=samples, logposts=logposts, accept_rates=acc, exchange_rates=xr)

    def run_mcmc(self, p, q, nsamples, nburnin=None, ntemperatures=None, nthin=1, seed=None, n_ensembles=1, priors=None):
        """CarmaModel.run_mcmc for every curve in one launch (carma_multi_pt_run), with the same defaults: curve c with
        the same seed gives what CarmaModel(curve c).run_mcmc gives when it is curve 0.  Returns a SurveySample (see
        carma_pack.survey_run_mcmc)."""
        from .carma_pack import survey_run_mcmc
        return survey_run_mcmc(self, p, q, nsamples, nburnin=nburnin, ntemperatures=ntemperatures, nthin=nthin, seed=seed,
                               n_ensembles=n_ensembles, priors=priors)

    def curve_stats(self):
        """Per-curve statistics (structured array, CURVE_STATS_DTYPE): y_mean, y_var_pop, y_var_sample, min_dt,
        median_dt, tspan, dt_max, ny."""
        out = np.empty(self.ncurves, dtype=CURVE_STATS_DTYPE)
        check(lib.carma_multi_series_curve_stats(self.handle, out.ctypes.data), "carma_multi_series_curve_stats")
        return out

    def mle_grid(self, jobs, priors=None, maxiter=1000, history=8, gtol=1e-5, ftol=2.2e-9, fd_eps=1e-8):
        """Every model of `jobs` fitted on every curve in one launch (carma_multi_mle_grid_device), the survey twin of
        Series.mle_grid.  jobs: sequence of (kind, p, q, x0, lower, upper, flags) with x0 (ncurves, nstart, d) and
        lower / upper (ncurves, d); priors: ncurves entries of PRIOR_DTYPE or None (population-variance defaults).
        Returns a list of (x (ncurves, nstart, d), f (ncurves, nstart), nit (ncurves,), nfev (ncurves,)), one per job."""
        nj, nc = len(jobs), self.ncurves
        cj = (MLEJob * max(nj, 1))()
        lo = np.zeros((max(nj, 1), nc, MAX_DIM))
        hi = np.zeros((max(nj, 1), nc, MAX_DIM))
        xs, shapes = [], []
        for j, (kind, p, q, x0, lower, upper, flags) in enumerate(jobs):
            d = model_dim(kind, p, q)
            x0 = np.ascontiguousarray(x0, dtype=np.float64)
            if x0.ndim != 3 or x0.shape[0] != nc or x0.shape[2] != d:
                raise ValueError("x0 of job %d must be (%d, nstart, %d)" % (j, nc, d))
            lo[j, :, :d] = np.broadcast_to(np.asarray(lower, dtype=np.float64), (nc, d))
            hi[j, :, :d] = np.broadcast_to(np.asarray(upper, dtype=np.float64), (nc, d))
            cj[j].kind, cj[j].p, cj[j].q, cj[j].flags, cj[j].nstart = kind, p, q, flags, x0.shape[1]
            xs.append(x0.reshape(-1))
            shapes.append((x0.shape[1], d))
        pp = None
        if priors is not None:
            priors = np.ascontiguousarray(priors, dtype=PRIOR_DTYPE)
            if priors.shape != (nc,):
                raise ValueError("priors must have %d entries" % nc)
            pp = priors.ctypes.data
        xin = np.ascontiguousarray(np.concatenate(xs)) if xs else np.zeros(0)
        xout = np.empty_like(xin)
        fout = np.empty(nc * sum(n for n, _ in shapes))
        nit = np.zeros((max(nj, 1), nc), dtype=np.intc)
        nfev = np.zeros((max(nj, 1), nc), dtype=np.longlong)
        o = MLEOpts()
        lib.carma_mle_default_opts(ctypes.byref(o))
        o.maxiter, o.history, o.gtol, o.ftol, o.fd_eps = int(maxiter), int(history), gtol, ftol, fd_eps
        check(lib.carma_multi_mle_grid_device(self.handle, nj, cj, pp, _ptr(xin), _ptr(lo), _ptr(hi), ctypes.byref(o),
                                              _ptr(xout), _ptr(fout), nit.ctypes.data_as(ctypes.POINTER(ctypes.c_int)),
                                              nfev.ctypes.data_as(ctypes.POINTER(ctypes.c_longlong))),
              "carma_multi_mle_grid_device")
        res, ox, of = [], 0, 0
        for j, (n, d) in enumerate(shapes):
            res.append((xout[ox:ox + nc * n * d].reshape(nc, n, d).copy(), fout[of:of + nc * n].reshape(nc, n).copy(),
                        nit[j].copy(), nfev[j].copy()))
            ox += nc * n * d
            of += nc * n
        return res

    def get_mle(self, p, q, ntrials=100, seed=None, maxiter=1000, curve_offset=0, priors=None):
        """CarmaModel.get_mle for every curve: one starting-value launch, then one fitting launch over all curves x
        starts.  Curve c's trial j is global trial (curve_offset + c) * ntrials + j, exactly as CarmaModel(curve
        c).get_mle(..., trial_offset=(curve_offset + c) * ntrials) numbers it, so a survey split into curve blocks gives
        the same fits.  Returns an OptimizeResult of per-curve arrays (see carma_pack.survey_get_mle)."""
        from .carma_pack import survey_get_mle
        return survey_get_mle(self, p, q, ntrials=ntrials, seed=seed, maxiter=maxiter, curve_offset=curve_offset,
                              priors=priors)

    def choose_order(self, pmax, qmax=None, pqlist=None, ntrials=100, seed=None, curve_offset=0):
        """CarmaModel.choose_order for every curve, all models x curves x starts in one fitting launch.  Returns
        (best_pq (ncurves, 2), pqlist, aicc (ncurves, nmodels), mles) (see carma_pack.survey_choose_order)."""
        from .carma_pack import survey_choose_order
        return survey_choose_order(self, pmax, qmax=qmax, pqlist=pqlist, ntrials=ntrials, seed=seed,
                                   curve_offset=curve_offset)

    def loglik_dev(self, kind, p, q, d_priors_ptr, d_theta_ptr, d_out_ptr, flags=0, stream=0):
        check(lib.carma_multi_loglik_dev(self.handle, kind, p, q, d_priors_ptr, d_theta_ptr, d_out_ptr, flags, stream),
              "carma_multi_loglik_dev")

    def _rows(self, kind, p, q, theta, priors):
        """theta (ncurves, d) and priors (ncurves entries or None) as contiguous arrays for the survey calls."""
        th = np.ascontiguousarray(theta, dtype=np.float64)
        d = model_dim(kind, p, q)
        if th.shape != (self.ncurves, d):
            raise ValueError("theta must be (%d, %d)" % (self.ncurves, d))
        if priors is not None:
            priors = np.ascontiguousarray(priors, dtype=PRIOR_DTYPE)
            if priors.shape != (self.ncurves,):
                raise ValueError("priors must have %d entries" % self.ncurves)
        return th, priors

    @staticmethod
    def _default_flags(p, flags):
        # the rule the survey fits use: SetMLE(True) only for p > 1 (carma_pack.py:242)
        return (0 if p == 1 else IGNORE_BOUNDS) if flags is None else flags

    def kalman_filter(self, kind, p, q, theta, priors=None, flags=None):
        """One-step predictive mean and variance of every point of every curve, one theta row per curve
        (carma_multi_filter, the survey form of CarmaSample.kalman_filter).  Returns (mean + mu, var, loglik): mean and
        var flat in the CSR order of the curves, loglik per curve (bitwise MultiSeries.loglik with the same arguments).
        flags: None = the survey fits' rule (0 for p == 1, else IGNORE_BOUNDS)."""
        th, priors = self._rows(kind, p, q, theta, priors)
        flags = self._default_flags(p, flags)
        total = int(self.offsets[-1])
        mean, var, ll = np.empty(total), np.empty(total), np.empty(self.ncurves)
        check(lib.carma_multi_filter(self.handle, kind, p, q, None if priors is None else priors.ctypes.data, th.ctypes.data,
                                     flags, mean.ctypes.data, var.ctypes.data, ll.ctypes.data), "carma_multi_filter")
        mean += np.repeat(th[:, 2], np.diff(self.offsets))
        return mean, var, ll

    def filter_dev(self, kind, p, q, d_priors_ptr, d_theta_ptr, d_mean_ptr, d_var_ptr, d_loglik_ptr=None, flags=None,
                   stream=0):
        """Device-resident kalman_filter (carma_multi_filter_dev): raw device pointers, mean without mu, no sync."""
        check(lib.carma_multi_filter_dev(self.handle, kind, p, q, d_priors_ptr, d_theta_ptr, self._default_flags(p, flags),
                                         d_mean_ptr, d_var_ptr, d_loglik_ptr, stream), "carma_multi_filter_dev")

    def assess_fit_values(self, kind, p, q, theta, nlags=20, priors=None, flags=None):
        """CarmaSample.assess_fit_values for every curve (carma_multi_assess_fit): moments and autocorrelation of the
        standardised one-step residuals, computed on the device.  Returns an OptimizeResult-style dict of per-curve arrays:
        loglik, resid_mean, resid_std, acf (ncurves, nlags), acf_sq (ncurves, nlags) -- lags 1..nlags -- and
        bound = 1.96 / sqrt(ny), the band a white residual stays in."""
        from .carma_pack import OptimizeResult
        th, priors = self._rows(kind, p, q, theta, priors)
        nlags = int(nlags)
        out = np.empty((self.ncurves, 3 + 2 * max(nlags, 0)))
        check(lib.carma_multi_assess_fit(self.handle, kind, p, q, None if priors is None else priors.ctypes.data,
                                         th.ctypes.data, self._default_flags(p, flags), nlags, out.ctypes.data),
              "carma_multi_assess_fit")
        return OptimizeResult(loglik=out[:, 0].copy(), resid_mean=out[:, 1].copy(), resid_std=out[:, 2].copy(),
                              acf=out[:, 3:3 + nlags].copy(), acf_sq=out[:, 3 + nlags:].copy(),
                              bound=1.96 / np.sqrt(np.diff(self.offsets).astype(np.float64)))

    def predict(self, kind, p, q, theta, tq, q_offsets, priors=None, flags=None):
        """Expected value and variance of every curve at its own query times given its data (carma_multi_predict, the
        survey form of CarmaSample.predict).  tq: absolute times, curve c's at tq[q_offsets[c]:q_offsets[c+1]], any
        order.  Returns (qmean + mu, qvar) in the order of tq."""
        th, priors = self._rows(kind, p, q, theta, priors)
        t = _c(np.atleast_1d(tq))
        qo = np.ascontiguousarray(q_offsets, dtype=np.int64)
        if qo.shape != (self.ncurves + 1,) or qo[-1] != t.size:
            raise ValueError("q_offsets must have %d entries and end at len(tq) = %d" % (self.ncurves + 1, t.size))
        qm, qv = np.empty(t.size), np.empty(t.size)
        check(lib.carma_multi_predict(self.handle, kind, p, q, None if priors is None else priors.ctypes.data, th.ctypes.data,
                                      self._default_flags(p, flags), qo.ctypes.data, t.ctypes.data, qm.ctypes.data,
                                      qv.ctypes.data), "carma_multi_predict")
        qm += np.repeat(th[:, 2], np.diff(qo))
        return qm, qv

    def conditional_simulate(self, kind, p, q, theta, tsim, s_offsets, npaths=1, seed=None, curve_offset=0, priors=None,
                             flags=None):
        """Draws of every curve at its own times given its data (carma_multi_simulate, the survey form of
        CarmaSample.simulate).  tsim: absolute times, curve c's at tsim[s_offsets[c]:s_offsets[c+1]], any order.
        theta: (ncurves, d), one row for all paths of a curve, or (ncurves, npaths, d), one row per path (posterior
        predictive).  Path j of curve c depends only on (seed, j, curve_offset + c) and its theta row.  Returns
        (npaths, len(tsim)) in the order of tsim, mu included.  flags: None = the survey fits' rule."""
        d = model_dim(kind, p, q)
        npaths = int(npaths)
        if npaths < 1:
            raise ValueError("npaths must be >= 1")
        th = np.ascontiguousarray(theta, dtype=np.float64)
        if th.shape == (self.ncurves, npaths, d):
            th = th.reshape(self.ncurves * npaths, d)
        elif th.shape != (self.ncurves, d):
            raise ValueError("theta must be (%d, %d) or (%d, %d, %d)" % (self.ncurves, d, self.ncurves, npaths, d))
        _, priors = self._rows(kind, p, q, th[:self.ncurves], priors)
        t = _c(np.atleast_1d(tsim))
        so = np.ascontiguousarray(s_offsets, dtype=np.int64)
        if so.shape != (self.ncurves + 1,) or so[0] != 0 or so[-1] != t.size:
            raise ValueError("s_offsets must have %d entries from 0 to len(tsim) = %d" % (self.ncurves + 1, t.size))
        if seed is None:
            seed = int(np.random.SeedSequence().generate_state(1, dtype=np.uint64)[0] >> 1)
        out = np.empty((npaths, t.size))
        check(lib.carma_multi_simulate(self.handle, kind, p, q, None if priors is None else priors.ctypes.data,
                                       th.ctypes.data, th.shape[0], self._default_flags(p, flags), so.ctypes.data,
                                       t.ctypes.data, npaths, int(seed), int(curve_offset), out.ctypes.data),
              "carma_multi_simulate")
        return out

    def smooth(self, kind, p, q, theta, tq=None, q_offsets=None, priors=None, flags=None, points=True):
        """Kalman smoother of every curve given all of its data (carma_multi_smooth): one pass forward and one backward,
        O(ny + nq) steps per curve.  theta, priors and flags as kalman_filter (flags None = the survey fits' rule).
        tq / q_offsets (optional, together): absolute query times as in predict.  Returns an OptimizeResult-style dict:
          mean, var          the noise-free process at every data point given the curve's data (flat, CSR, mu included);
          loo_mean, loo_var  the law of each y given every other point of its curve (mu and measurement noise included):
                             (y - loo_mean) / sqrt(loo_var) is the standardised deleted residual, for flagging outliers;
          loglik             per curve, bitwise MultiSeries.loglik;
          qmean, qvar        the smoothed process at tq, in the order of tq (only when tq is given).
        points=False leaves out the four per-point arrays (nothing but loglik and the queries crosses PCIe), for a caller
        who only wants the curves on a grid.  A row outside the prior gives NaN for its curve and -inf loglik."""
        from .carma_pack import OptimizeResult
        th, priors = self._rows(kind, p, q, theta, priors)
        if (tq is None) != (q_offsets is None):
            raise ValueError("tq and q_offsets must be given together")
        qo = t = None
        if tq is not None:
            t = _c(np.atleast_1d(tq))
            qo = np.ascontiguousarray(q_offsets, dtype=np.int64)
            if qo.shape != (self.ncurves + 1,) or qo[0] != 0 or qo[-1] != t.size:
                raise ValueError("q_offsets must have %d entries from 0 to len(tq) = %d" % (self.ncurves + 1, t.size))
        total = int(self.offsets[-1]) if points else 0
        mean, var, lm, lv, ll = np.empty(total), np.empty(total), np.empty(total), np.empty(total), np.empty(self.ncurves)
        ptr = (lambda a: a.ctypes.data) if points else (lambda a: None)
        qm = qv = None
        if t is not None:
            qm, qv = np.empty(t.size), np.empty(t.size)
        check(lib.carma_multi_smooth(self.handle, kind, p, q, None if priors is None else priors.ctypes.data, th.ctypes.data,
                                     self._default_flags(p, flags), ptr(mean), ptr(var), ptr(lm), ptr(lv), ll.ctypes.data,
                                     None if qo is None else qo.ctypes.data,
                                     None if t is None else t.ctypes.data, None if qm is None else qm.ctypes.data,
                                     None if qv is None else qv.ctypes.data), "carma_multi_smooth")
        res = OptimizeResult(loglik=ll)
        if points:
            mu = np.repeat(th[:, 2], np.diff(self.offsets))
            res.update(mean=mean + mu, var=var, loo_mean=lm + mu, loo_var=lv)
        if t is not None:
            res.qmean = qm + np.repeat(th[:, 2], np.diff(qo))
            res.qvar = qv
        return res

    def hessian(self, kind, p, q, theta, priors=None, flags=None, rel_step=None):
        """Gradient, Hessian and Laplace covariance of every curve's log-density at its theta row
        (carma_multi_hessian): central finite differences, d^2 + d + 1 evaluations per curve in one launch.  The
        function is exactly MultiSeries.loglik with the same priors and flags (None = the survey fits' rule), so at a
        fit, hessian(kind, p, q, fit.x).loglik is -fit.fun.  Steps h_i = rel_step * (theta_0, theta_1, theta_0, 1, ...)_i
        (rel_step None or <= 0: HESS_REL_STEP = 2^-13).  Returns an OptimizeResult-style dict:
          loglik (nc,), grad (nc, d), hessian (nc, d, d), cov (nc, d, d) = (-hessian)^-1,
          stderr (nc, d) = sqrt(diag(cov)), NaN unless status is HESS_OK,
          status (nc,) one of HESS_OK, HESS_REJECTED (loglik -inf, the rest NaN), HESS_NONFINITE (a stencil value is
          not finite: grad / hessian / cov NaN), HESS_NOT_NEGDEF (-hessian not positive definite: cov NaN),
          step (nc, d) the h used."""
        from .carma_pack import OptimizeResult
        th, priors = self._rows(kind, p, q, theta, priors)
        rs = HESS_REL_STEP if rel_step is None else float(rel_step)
        if not np.isfinite(rs):
            raise ValueError("rel_step must be finite")
        if rs <= 0.0:
            rs = HESS_REL_STEP
        nc, d = self.ncurves, th.shape[1]
        ll, g, h, cov = np.empty(nc), np.empty((nc, d)), np.empty((nc, d, d)), np.empty((nc, d, d))
        st = np.empty(nc, dtype=np.intc)
        check(lib.carma_multi_hessian(self.handle, kind, p, q, None if priors is None else priors.ctypes.data,
                                      th.ctypes.data, self._default_flags(p, flags), rs, ll.ctypes.data, g.ctypes.data,
                                      h.ctypes.data, cov.ctypes.data, st.ctypes.data), "carma_multi_hessian")
        stderr = np.sqrt(np.diagonal(cov, axis1=1, axis2=2))
        stderr = np.where((st == HESS_OK)[:, None], stderr, np.nan)
        return OptimizeResult(loglik=ll, grad=g, hessian=h, cov=cov, stderr=stderr, status=st.astype(np.int64),
                              step=hessian_steps(th, rs))

    def laplace(self, kind, p, q, theta, cov, ndraws=1000, seed=None, curve_offset=0, priors=None, flags=0):
        """Importance sampling of every curve's posterior from its Laplace approximation N(theta_c, cov_c)
        (carma_multi_laplace): ndraws draws per curve, each draw's exact log-density, the Pareto k-hat of the weights and
        an equally weighted resample, in one call.  The target is MultiSeries.loglik with these priors (None: the
        population-variance defaults) and flags.  The defaults, flags 0 and those priors, are the posterior run_mcmc
        samples, so that the weights target it; they differ from hessian's default (the survey fits' rule, which skips
        the prior bounds for p > 1), because a fit's curvature and a posterior's draws answer different questions.
        Draw j of curve c depends only on (seed, j, curve_offset + c, theta_c, cov_c).  Returns an OptimizeResult-style
        dict:
          draws (nc, ndraws, d), logpost (nc, ndraws) bitwise MultiSeries.loglik of the draws, logq (nc, ndraws) the
          proposal's log-density, log_weights = logpost - logq (-inf where logpost is not finite; NaN for
          every draw of a LAPLACE_BAD_COV curve, which has no draws),
          ess (nc,) the weight ESS, khat (nc,) the Pareto k-hat (<= 0.7: the Gaussian answer is good; above: run MCMC),
          resample (nc, ndraws) indices into draws of an equally weighted sample (-1 unless status is LAPLACE_OK),
          status (nc,) one of LAPLACE_OK, LAPLACE_BAD_COV (cov or theta not finite, or not positive definite: NaN
          draws), LAPLACE_NO_WEIGHT (no draw has a finite logpost)."""
        from .carma_pack import OptimizeResult
        th, priors = self._rows(kind, p, q, theta, priors)
        nc, d = self.ncurves, th.shape[1]
        cv = np.ascontiguousarray(cov, dtype=np.float64)
        if cv.shape != (nc, d, d):
            raise ValueError("cov must be (%d, %d, %d)" % (nc, d, d))
        S = int(ndraws)
        if not 1 <= S <= LAPLACE_MAX_DRAWS:
            raise ValueError("ndraws must be in 1 .. %d" % LAPLACE_MAX_DRAWS)
        curve_offset = int(curve_offset)
        if curve_offset < 0 or curve_offset + nc > 2 ** 32:
            raise ValueError("curve_offset must be >= 0 with curve_offset + ncurves <= 2^32")
        if seed is None:
            seed = int(np.random.SeedSequence().generate_state(1, dtype=np.uint64)[0] >> 1)
        draws, lp, lq = np.empty((nc, S, d)), np.empty((nc, S)), np.empty((nc, S))
        rs = np.empty((nc, S), dtype=np.int32)
        ess, kh, st = np.empty(nc), np.empty(nc), np.empty(nc, dtype=np.intc)
        check(lib.carma_multi_laplace(self.handle, kind, p, q, None if priors is None else priors.ctypes.data,
                                      th.ctypes.data, cv.ctypes.data, int(flags), S, int(seed), curve_offset,
                                      draws.ctypes.data, lp.ctypes.data, lq.ctypes.data, rs.ctypes.data, ess.ctypes.data,
                                      kh.ctypes.data, st.ctypes.data), "carma_multi_laplace")
        lw = np.where(np.isfinite(lp), lp - lq, -np.inf)
        lw[st == LAPLACE_BAD_COV] = np.nan
        return OptimizeResult(draws=draws, logpost=lp, logq=lq, log_weights=lw, ess=ess, khat=kh, resample=rs,
                              status=st.astype(np.int64))

    def laplace_sample(self, p, q, theta, cov=None, ndraws=1000, seed=None, curve_offset=0, priors=None):
        """The posterior of every curve by importance sampling from its Laplace approximation at theta (e.g.
        get_mle(p, q).x): laplace() with run_mcmc's posterior, resampled to an equally weighted sample.  cov None: the
        covariance of hessian(kind, p, q, theta, priors=priors); a curve whose Hessian status is not HESS_OK comes back
        LAPLACE_BAD_COV.  Returns a LaplaceSample (a SurveySample: derived parameters, psd_credible_band, map_theta, DIC
        and curve(c) work as for run_mcmc's) with khat, ess, status and the raw laplace() result; the trace rows of a
        curve whose status is not LAPLACE_OK are NaN, so its summaries are NaN."""
        from .carma_pack import LaplaceSample, _kind_for
        if not p > q:
            raise ValueError("Order of AR polynomial, p, must be larger than order of MA polynomial, q.")
        kind = _kind_for(p, q)
        th, priors = self._rows(kind, p, q, theta, priors)
        if cov is None:
            h = self.hessian(kind, p, q, th, priors=priors)
            cov = np.where((h.status == HESS_OK)[:, None, None], h.cov, np.nan)
        r = self.laplace(kind, p, q, th, cov, ndraws=ndraws, seed=seed, curve_offset=curve_offset, priors=priors)
        nc = self.ncurves
        idx = np.maximum(r.resample, 0)
        trace = r.draws[np.arange(nc)[:, None], idx]
        lp = r.logpost[np.arange(nc)[:, None], idx]
        bad = r.status != LAPLACE_OK
        trace[bad] = np.nan
        lp[bad] = np.nan
        if priors is None:
            priors = self.default_priors(population_var=True)
        return LaplaceSample(trace, lp, p, q, r, kind=kind, priors=priors, stats=self.curve_stats(), multi_series=self)


def hessian_steps(theta, rel_step=HESS_REL_STEP):
    """The finite-difference steps of carma_multi_hessian for theta rows (n, d): rel_step * (theta_0, theta_1, theta_0,
    1, 1, ...), each one rounded product."""
    th = np.atleast_2d(np.asarray(theta, dtype=np.float64))
    s = np.ones_like(th)
    s[:, 0], s[:, 1], s[:, 2] = th[:, 0], th[:, 1], th[:, 0]
    return rel_step * s


def lbfgs_batch(fun_batch, x0, lower, upper, maxiter=1000, history=8, gtol=1e-5, ftol=2.2e-9, fd_eps=1e-8):
    """The native optimiser core (carma_lbfgs_batch) on a Python objective: fun_batch maps an (n, d) array to n
    values.  Host code only; this is the loop Series.mle_batch runs with the GPU log-density as objective."""
    x0 = np.ascontiguousarray(x0, dtype=np.float64)
    n, d = x0.shape
    lo, hi = _c(np.broadcast_to(lower, (d,))), _c(np.broadcast_to(upper, (d,)))

    def trampoline(theta, npts, dim, fout, _user):
        try:
            th = np.ctypeslib.as_array(theta, shape=(npts, dim))
            np.ctypeslib.as_array(fout, shape=(npts,))[:] = np.asarray(fun_batch(th.copy()), dtype=np.float64)
            return 0
        except Exception:  # noqa: BLE001
            return 1

    cb = OBJECTIVE_FN(trampoline)
    o = MLEOpts()
    lib.carma_mle_default_opts(ctypes.byref(o))
    o.maxiter, o.history, o.gtol, o.ftol, o.fd_eps = int(maxiter), int(history), gtol, ftol, fd_eps
    x, f = np.empty((n, d)), np.empty(n)
    nit, nfev = ctypes.c_int(0), ctypes.c_longlong(0)
    check(lib.carma_lbfgs_batch(cb, None, d, n, _ptr(x0), _ptr(lo), _ptr(hi), ctypes.byref(o), _ptr(x), _ptr(f),
                                ctypes.byref(nit), ctypes.byref(nfev)), "carma_lbfgs_batch")
    return x, f, nit.value, nfev.value


def log_prior(kind, p, theta, prior):
    th = _c(theta)
    out = ctypes.c_double()
    check(lib.carma_log_prior(kind, p, _ptr(th), ctypes.byref(prior), ctypes.byref(out)), "carma_log_prior")
    return out.value


def fp64_peak_tflops(device=0):
    out = ctypes.c_double()
    check(lib.carma_fp64_peak_tflops(device, ctypes.byref(out)), "carma_fp64_peak_tflops")
    return out.value


def philox_dev(c0, c1, c2, c3, seed):
    out = (ctypes.c_uint32 * 4)()
    check(lib.carma_philox_dev(c0, c1, c2, c3, seed, out), "carma_philox_dev")
    return [int(x) for x in out]


def tdist_dev(seed, chain, it, j, dof=8):
    out = ctypes.c_double()
    check(lib.carma_tdist_dev(seed, chain, it, j, dof, ctypes.byref(out)), "carma_tdist_dev")
    return out.value


def fastmath_dev(rate, dt):
    """The time loop's transcendentals (csrc/fast_math.cuh) on arrays: rate in table steps per unit time.
    Returns exp(rate dt ln2/64), sin and cos(rate dt pi/64), (1-rho)/2 and (1+rho)/2 with rho = the exponential, 1/rate."""
    rate, dt = _c(rate), _c(dt)
    outs = [np.empty(rate.size) for _ in range(6)]
    check(lib.carma_fastmath_dev(_ptr(rate), _ptr(dt), rate.size, *[_ptr(o) for o in outs]), "carma_fastmath_dev")
    return tuple(outs)
