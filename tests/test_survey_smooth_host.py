"""CPU-side checks of carma_multi_smooth / MultiSeries.smooth.

  * the entry point rejects a null handle, null theta and query offsets that do not start at 0 with CARMA_ERR_ARG and a
    message naming it, before any CUDA call; the binding is exported and declared;
  * MultiSeries.smooth checks its arguments before it uses the handle;
  * the per-curve recursion multi_smooth_kernel runs (smooth_forward / smooth_backward in kalman_real.cuh, compiled here
    for the host by tests/host_check/smoothcheck.cu) agrees with the dense Gaussian-process conditional: smoothed mean
    and variance at the data times and at query times, and the leave-one-out law of every point."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import build_native
from carma_pack_b200 import synth
from oracle import oracle as O

CARMA_ERR_ARG = 1
HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "host_check", "smoothcheck.cu")
LIB = os.path.join(HERE, "host_check", "libsmoothcheck.so")
CSRC = os.path.join(os.path.dirname(HERE), "carma_pack_b200", "csrc")
_dp = ctypes.POINTER(ctypes.c_double)


def test_survey_smooth_rejects_bad_arguments_before_cuda():
    import carma_pack_b200 as C
    L = C._lib.lib
    th = np.zeros(8)
    qo = np.array([0, 2, 3], dtype=np.int64)
    tq = np.zeros(3)
    out = np.zeros(16)

    def call(m=None, theta=th.ctypes.data, offs=qo.ctypes.data):
        return L.carma_multi_smooth(m, C.KIND_CARMA, 3, 1, None, theta, 0, out.ctypes.data, None, None, None, None, offs,
                                    tq.ctypes.data, None, None)

    for kw in ({}, {"theta": None}, {"offs": None}):
        assert call(**kw) == CARMA_ERR_ARG
        assert b"carma_multi_smooth" in L.carma_last_error() and b"null" in L.carma_last_error()
    bad = np.array([1, 2, 3], dtype=np.int64)
    assert call(offs=bad.ctypes.data) == CARMA_ERR_ARG
    assert b"carma_multi_smooth" in L.carma_last_error() and b"q_offsets" in L.carma_last_error()


def test_survey_smooth_binding_is_declared():
    import carma_pack_b200 as C
    assert "carma_multi_smooth" in C._lib.EXPORTED_SYMBOLS
    assert C._lib.lib.carma_multi_smooth.argtypes is not None and len(C._lib.lib.carma_multi_smooth.argtypes) == 16
    assert callable(C.MultiSeries.smooth)


def test_smooth_argument_errors_raise_value_error():
    """The shape checks run before the handle is used, so an object without one shows them."""
    import carma_pack_b200 as C
    fake = object.__new__(C.MultiSeries)
    fake.ncurves = 2
    fake.offsets = np.array([0, 3, 6], dtype=np.int64)
    fake.handle = None
    d = C._lib.model_dim(C.KIND_CARMA, 3, 1)
    th = np.zeros((2, d))
    tq = np.arange(4.0)
    with pytest.raises(ValueError, match="theta"):
        fake.smooth(C.KIND_CARMA, 3, 1, np.zeros((3, d)))
    with pytest.raises(ValueError, match="together"):
        fake.smooth(C.KIND_CARMA, 3, 1, th, tq=tq)
    with pytest.raises(ValueError, match="together"):
        fake.smooth(C.KIND_CARMA, 3, 1, th, q_offsets=[0, 2, 4])
    for qo in ([0, 2], [0, 2, 5], [1, 2, 4]):
        with pytest.raises(ValueError, match="q_offsets"):
            fake.smooth(C.KIND_CARMA, 3, 1, th, tq=tq, q_offsets=qo)
    with pytest.raises(ValueError, match="priors"):
        fake.smooth(C.KIND_CARMA, 3, 1, th, priors=np.zeros(3, dtype=C._lib.PRIOR_DTYPE))


# ---- the recursion on the host against the dense GP conditional ----------------------------------------------------

@pytest.fixture(scope="module")
def H():
    deps = [SRC] + [os.path.join(CSRC, f) for f in ("kalman_real.cuh", "fast_math.cuh", "theta_transform.cuh", "device_math.cuh")]
    if not (os.path.exists(LIB) and all(os.path.getmtime(LIB) >= os.path.getmtime(d) for d in deps)):
        subprocess.check_call([build_native.NVCC, "-O2", "-std=c++17", "-Xcompiler", "-fPIC", "-shared",
                               "--expt-relaxed-constexpr", "-Wno-deprecated-gpu-targets", "-o", LIB, SRC],
                              stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    L = ctypes.CDLL(LIB)
    L.smoothcheck.restype = ctypes.c_int
    return L


def host_smooth(L, kind, p, q, t, y, e, theta, prior, tq, flags=1):
    t, y, e, th, tq = (np.ascontiguousarray(a, float) for a in (t, y, e, theta, tq))
    out = np.empty(4 * t.size + 1)
    qm, qv = np.empty(tq.size), np.empty(tq.size)
    rc = L.smoothcheck(kind, p, q, ctypes.c_uint(flags), ctypes.byref(prior), t.ctypes.data_as(_dp), y.ctypes.data_as(_dp),
                       e.ctypes.data_as(_dp), ctypes.c_size_t(t.size), th.ctypes.data_as(_dp), tq.ctypes.data_as(_dp),
                       ctypes.c_size_t(tq.size), out.ctypes.data_as(_dp), qm.ctypes.data_as(_dp), qv.ctypes.data_as(_dp))
    assert rc == 0
    n = t.size
    return out[:n], out[n:2 * n], out[2 * n:3 * n], out[3 * n:4 * n], out[4 * n], qm, qv


def dense_gp(kind, p, q, t, y, e, theta, prior, tq):
    """Smoothed mean / var at t and tq, and the leave-one-out law of y, from the dense covariance (means without mu)."""
    roots = O.ar_roots(np.asarray(theta[3:3 + p]))
    ma = O.ma_coefs(kind, np.asarray(theta, float), p, q, prior)
    v1 = synth.carma_variance(1.0, roots, ma)
    cov = lambda lag: theta[0] ** 2 * synth.carma_variance(1.0, roots, ma, lag=lag) / v1   # noqa: E731
    Kf = cov(np.abs(t[:, None] - t[None, :]))
    K = Kf + np.diag(theta[1] * e ** 2)
    Ki = np.linalg.inv(K)
    r = y - theta[2]
    a = Ki @ r
    mean = Kf @ a
    var = np.diag(Kf - Kf @ Ki @ Kf)
    loo_mean = r - a / np.diag(Ki)
    loo_var = 1.0 / np.diag(Ki)
    ks = cov(np.abs(tq[:, None] - t[None, :]))
    qmean = ks @ a
    qvar = theta[0] ** 2 - np.einsum("ij,jk,ik->i", ks, Ki, ks)
    return mean, var, loo_mean, loo_var, qmean, qvar


def _logquad(roots):
    return list(synth.roots_to_logquad(roots))


HOST_MODELS = [
    ("carma10", 1, 0, _logquad([-0.3])),
    ("carma20", 2, 0, _logquad([-0.1 + 0.5j, -0.1 - 0.5j])),
    ("carma31_conj", 3, 1, _logquad([-0.05 + 0.3j, -0.05 - 0.3j, -0.4]) + [np.log(2.0)]),
    ("carma31_real", 3, 1, _logquad([-0.1, -0.7, -0.3]) + [np.log(2.0)]),
    ("carma53", 5, 3, _logquad([-0.05 + 0.3j, -0.05 - 0.3j, -0.2, -0.9, -0.4]) + _logquad([-1.5 + 0.5j, -1.5 - 0.5j, -3.0])),
]


@pytest.mark.parametrize("model", range(len(HOST_MODELS)))
def test_host_recursion_matches_dense_gp(H, model):
    name, p, q, tail = HOST_MODELS[model]
    kind = O.KIND_CARMA
    rng = np.random.default_rng(40 + model)
    ar, ma, s2 = synth.carma31_truth()
    ny = 60
    t = np.cumsum(rng.uniform(0.2, 3.0, ny)) + 7.0
    y = 2.0 + synth.carma_process(t, s2, ar, ma, rng) + 0.2 * rng.standard_normal(ny)
    e = rng.uniform(0.1, 0.3, ny)
    theta = np.array([np.std(y), 1.1, np.mean(y)] + list(tail))
    prior = O.default_prior(t, y)
    span = t[-1] - t[0]
    tq = np.concatenate([[t[0] - 0.5 * span, t[0] - 1e-3, t[0], t[17], t[17], t[-1], t[-1] + 2.0, t[-1] + span],
                         rng.uniform(t[0], t[-1], 15)])
    tq = tq[rng.permutation(tq.size)]
    mean, var, lm, lv, ll, qm, qv = host_smooth(H, kind, p, q, t, y, e, theta, prior, tq)
    dm, dv, dlm, dlv, dqm, dqv = dense_gp(kind, p, q, t, y, e, theta, prior, tq)
    sy, v0 = np.std(y), theta[0] ** 2
    np.testing.assert_allclose(mean, dm, rtol=0, atol=1e-9 * sy, err_msg=name)
    np.testing.assert_allclose(var, dv, rtol=1e-7, atol=1e-8 * v0, err_msg=name)
    np.testing.assert_allclose(lm, dlm, rtol=0, atol=1e-9 * sy, err_msg=name)
    np.testing.assert_allclose(lv, dlv, rtol=1e-7, atol=1e-8 * v0, err_msg=name)
    np.testing.assert_allclose(qm, dqm, rtol=0, atol=1e-9 * sy, err_msg=name)
    np.testing.assert_allclose(qv, dqv, rtol=1e-7, atol=1e-8 * v0, err_msg=name)
    # the log-density of the same recursion is the oracle's
    want = O.logdensity(kind, p, q, t, y, e, theta[None, :], prior=prior, ignore_prior=True)[0]
    np.testing.assert_allclose(ll, want, rtol=1e-9)
