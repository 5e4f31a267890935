"""CPU-side checks of carma_multi_laplace / MultiSeries.laplace / laplace_sample.

  * the entry point rejects null m / theta / cov, an invalid (kind, p, q) and ndraws 0 or above
    CARMA_LAPLACE_MAX_DRAWS with CARMA_ERR_ARG and a message naming it, before any CUDA call (curve_offset + ncurves
    > 2^32 needs a multi-series, so tests/test_gpu_survey_laplace.py checks it); the binding is exported and declared, and the Python calls check shapes and ranges before they use the handle;
  * the per-curve arithmetic of laplace.cuh, compiled here for the host by tests/host_check/laplacecheck.cu, is the
    documented one: the Cholesky factor is numpy's transcription of the documented loop bit for bit, and the weight ESS,
    the Pareto k-hat (ArviZ's _psislw / _gpdfit with r_eff = 1, written out below) and the systematic resample agree with
    numpy; on Pareto-tailed synthetic weights k-hat lands near the true shape."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import build_native

CARMA_ERR_ARG = 1
HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "host_check", "laplacecheck.cu")
LIB = os.path.join(HERE, "host_check", "liblaplacecheck.so")
CSRC = os.path.join(os.path.dirname(HERE), "carma_pack_b200", "csrc")
_dp = ctypes.POINTER(ctypes.c_double)


# ---- numpy references of the documented formulas (include/carma_b200.h, carma_multi_laplace) ----------------------

def chol_reference(cov):
    """The documented factorisation in numpy, loop for loop: lower triangle only, every product and difference rounded
    on its own.  Returns (L, log|L|) or (None, None) where a pivot is not positive."""
    d = cov.shape[0]
    L = np.zeros((d, d))
    for j in range(d):
        s = cov[j, j]
        for k in range(j):
            s = s - L[j, k] * L[j, k]
        if not (s > 0.0) or not np.isfinite(s):
            return None, None
        L[j, j] = np.sqrt(s)
        for i in range(j + 1, d):
            t = cov[i, j]
            for k in range(j):
                t = t - L[i, k] * L[j, k]
            L[i, j] = t / L[j, j]
    return L, float(np.sum(np.log(np.diag(L))))


def gpdfit_reference(x):
    """ArviZ's _gpdfit on the ascending tail x: the k-hat of (n k + 5) / (n + 10)."""
    n = x.size
    m = 30 + int(n ** 0.5)
    b = 1.0 - np.sqrt(m / (np.arange(1, m + 1, dtype=float) - 0.5))
    b /= 3.0 * x[int(n / 4 + 0.5) - 1]
    b += 1.0 / x[-1]
    k = np.log1p(-b[:, None] * x).mean(axis=1)
    L = n * (np.log(-(b / k)) - k - 1.0)
    w = 1.0 / np.exp(L - L[:, None]).sum(axis=1)
    keep = w >= 10.0 * np.finfo(float).eps
    w, b = w[keep], b[keep]
    w /= w.sum()
    bbar = np.sum(b * w)
    kk = np.log1p(-bbar * x).mean()
    return (n * kk + 5.0) / (n + 10.0)


def khat_reference(lw):
    """ArviZ's _psislw k-hat (r_eff = 1) of the log weights lw."""
    S = lw.size
    a = lw - lw.max()
    if S < 2:
        return np.inf
    M = int(np.ceil(min(0.2 * S, 3.0 * np.sqrt(S))))
    cut = max(np.sort(a)[S - M - 1], np.log(np.finfo(float).tiny))
    tail = a[a > cut]
    if tail.size <= 4:
        return np.inf
    return gpdfit_reference(np.sort(np.exp(tail) - np.exp(cut)))


def ess_reference(lw):
    e = np.exp(lw - lw.max())
    return e.sum() ** 2 / (e ** 2).sum()


def resample_reference(lw, u):
    """Systematic resampling: index i -> the first j with C_j > ((i + u) / S) T (capped at S - 1), and the distance of
    each target to the nearest running sum relative to T (where the device's summation order may decide it)."""
    S = lw.size
    C = np.cumsum(np.exp(lw - lw.max()))
    T = C[-1]
    tgt = (np.arange(S) + u) / S * T
    idx = np.minimum(np.searchsorted(C, tgt, side="right"), S - 1)
    near = np.min(np.abs(C[None, :] - tgt[:, None]), axis=1) / T if S <= 4096 else None
    return idx, near


# ---- argument checks ----------------------------------------------------------------------------------------------

def test_survey_laplace_rejects_bad_arguments_before_cuda():
    import carma_pack_b200 as C
    L = C._lib.lib
    th, cov = np.zeros(7), np.eye(7)
    out = np.zeros(64)

    def call(m=None, kind=C.KIND_CARMA, p=3, q=1, theta=th.ctypes.data, cv=cov.ctypes.data, ndraws=10, off=0):
        return L.carma_multi_laplace(m, kind, p, q, None, theta, cv, 0, ndraws, 1, off, out.ctypes.data, None, None,
                                     None, None, None, None)

    assert call() == CARMA_ERR_ARG
    assert b"carma_multi_laplace" in L.carma_last_error() and b"null" in L.carma_last_error()
    fake = ctypes.c_void_p(1)   # never dereferenced: theta / cov are checked first
    assert call(m=fake, theta=None) == CARMA_ERR_ARG and b"null" in L.carma_last_error()
    assert call(m=fake, cv=None) == CARMA_ERR_ARG and b"null" in L.carma_last_error()
    for kind, p, q in ((C.KIND_CARMA, 3, 3), (C.KIND_CARMA, 0, 0), (C.KIND_CARMA, 8, 1), (9, 2, 0)):
        assert call(m=fake, kind=kind, p=p, q=q) == CARMA_ERR_ARG
        assert b"carma_multi_laplace" in L.carma_last_error() and b"invalid" in L.carma_last_error()
    for n in (0, C.LAPLACE_MAX_DRAWS + 1, 2 ** 40):
        assert call(m=fake, ndraws=n) == CARMA_ERR_ARG
        assert b"ndraws" in L.carma_last_error()


def test_survey_laplace_binding_is_declared():
    import carma_pack_b200 as C
    assert "carma_multi_laplace" in C._lib.EXPORTED_SYMBOLS
    at = C._lib.lib.carma_multi_laplace.argtypes
    assert at is not None and len(at) == 18 and at[8] is ctypes.c_size_t and at[9] is ctypes.c_uint64
    assert at[10] is ctypes.c_uint32
    assert (C.LAPLACE_OK, C.LAPLACE_BAD_COV, C.LAPLACE_NO_WEIGHT) == (0, 1, 2) and C.LAPLACE_MAX_DRAWS == 2 ** 20
    assert callable(C.MultiSeries.laplace) and callable(C.MultiSeries.laplace_sample)
    assert callable(C.CarmaModel.laplace_sample) and issubclass(C.LaplaceSample, C.SurveySample)
    hdr = open(os.path.join(os.path.dirname(HERE), "include", "carma_b200.h")).read()
    assert "#define CARMA_LAPLACE_MAX_DRAWS (1u << 20)" in hdr
    assert "CARMA_LAPLACE_OK = 0, CARMA_LAPLACE_BAD_COV = 1, CARMA_LAPLACE_NO_WEIGHT = 2" in hdr


def test_laplace_argument_errors_raise_value_error():
    """The shape and range checks run before the handle is used, so an object without one shows them."""
    import carma_pack_b200 as C
    fake = object.__new__(C.MultiSeries)
    fake.ncurves = 2
    fake.offsets = np.array([0, 3, 6], dtype=np.int64)
    fake.handle = None
    d = C._lib.model_dim(C.KIND_CARMA, 3, 1)
    th, cov = np.ones((2, d)), np.tile(np.eye(d), (2, 1, 1))
    with pytest.raises(ValueError, match="theta"):
        fake.laplace(C.KIND_CARMA, 3, 1, np.zeros((3, d)), cov)
    with pytest.raises(ValueError, match="cov"):
        fake.laplace(C.KIND_CARMA, 3, 1, th, np.zeros((2, d, d + 1)))
    with pytest.raises(ValueError, match="cov"):
        fake.laplace(C.KIND_CARMA, 3, 1, th, np.zeros((1, d, d)))
    with pytest.raises(ValueError, match="priors"):
        fake.laplace(C.KIND_CARMA, 3, 1, th, cov, priors=np.zeros(3, dtype=C._lib.PRIOR_DTYPE))
    for n in (0, C.LAPLACE_MAX_DRAWS + 1):
        with pytest.raises(ValueError, match="ndraws"):
            fake.laplace(C.KIND_CARMA, 3, 1, th, cov, ndraws=n)
    for off in (-1, 2 ** 32 - 1):
        with pytest.raises(ValueError, match="curve_offset"):
            fake.laplace(C.KIND_CARMA, 3, 1, th, cov, curve_offset=off)
    with pytest.raises(ValueError, match="theta"):
        fake.laplace_sample(3, 1, np.zeros((2, d + 1)), cov=cov)
    with pytest.raises(ValueError, match="AR polynomial"):
        fake.laplace_sample(1, 1, th, cov=cov)


def test_laplace_sample_refuses_autocorrelation_ess():
    import carma_pack_b200 as C
    r = C.carma_pack.OptimizeResult(khat=np.zeros(1), ess=np.ones(1), status=np.zeros(1, dtype=np.int64))
    s = C.LaplaceSample(np.zeros((1, 5, 4)), np.zeros((1, 5)), 1, 0, r)
    with pytest.raises(ValueError, match=r"\.ess"):
        s.effective_samples("mu")


# ---- the per-curve arithmetic on the host -------------------------------------------------------------------------

@pytest.fixture(scope="module")
def H():
    deps = [SRC] + [os.path.join(CSRC, f) for f in ("laplace.cuh", "theta_transform.cuh", "fast_math.cuh", "device_math.cuh")]
    if not (os.path.exists(LIB) and all(os.path.getmtime(LIB) >= os.path.getmtime(d) for d in deps)):
        subprocess.check_call([build_native.NVCC, "-O2", "-std=c++17", "-Xcompiler", "-fPIC", "-shared",
                               "--expt-relaxed-constexpr", "-Wno-deprecated-gpu-targets", "-o", LIB, SRC],
                              stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    L = ctypes.CDLL(LIB)
    L.lap_chol_host.argtypes = [ctypes.c_int, _dp, _dp, _dp, _dp]
    L.lap_summary_host.argtypes = [_dp, ctypes.c_size_t, ctypes.c_double, _dp, _dp, ctypes.POINTER(ctypes.c_int)]
    return L


def host_chol(H, centre, cov):
    d = centre.size
    centre, cov = np.ascontiguousarray(centre, float), np.ascontiguousarray(cov, float)
    L, ld = np.empty((d, d)), ctypes.c_double()
    st = H.lap_chol_host(d, centre.ctypes.data_as(_dp), cov.ctypes.data_as(_dp), L.ctypes.data_as(_dp), ctypes.byref(ld))
    return st, L, ld.value


def host_summary(H, lw, u):
    lw = np.ascontiguousarray(lw, float)
    ess, kh = ctypes.c_double(), ctypes.c_double()
    rs = np.empty(lw.size, dtype=np.intc)
    st = H.lap_summary_host(lw.ctypes.data_as(_dp), lw.size, u, ctypes.byref(ess), ctypes.byref(kh),
                            rs.ctypes.data_as(ctypes.POINTER(ctypes.c_int)))
    return st, ess.value, kh.value, rs


@pytest.mark.parametrize("d", [1, 4, 7, 16])
def test_host_cholesky_is_the_documented_loop(H, d):
    rng = np.random.default_rng(d)
    A = rng.normal(size=(d, d))
    cov = A @ A.T + 0.1 * np.eye(d)
    cov[np.triu_indices(d, 1)] = 7.0            # the upper triangle is never read
    st, L, ld = host_chol(H, np.zeros(d), cov)
    want, wld = chol_reference(cov)
    assert st == 0
    np.testing.assert_array_equal(L, want)
    assert abs(ld - wld) <= 1e-14 * max(1.0, abs(wld))
    low = np.tril(cov) + np.tril(cov, -1).T
    np.testing.assert_allclose(L @ L.T, low, rtol=0, atol=1e-13 * np.abs(low).max())


def test_host_cholesky_status(H):
    d = 4
    cov = np.eye(d)
    assert host_chol(H, np.zeros(d), cov)[0] == 0
    for bad in ((np.nan, 2, 1), (np.inf, 3, 3)):
        c = cov.copy()
        c[bad[1], bad[2]] = bad[0]
        st, L, ld = host_chol(H, np.zeros(d), c)
        assert st == 1 and np.all(np.isnan(L)) and np.isnan(ld)
    c = cov.copy()
    c[0, 3] = np.nan                             # upper triangle: not read
    assert host_chol(H, np.zeros(d), c)[0] == 0
    c = cov.copy()
    c[2, 1] = c[1, 2] = 1.5                      # not positive definite
    assert host_chol(H, np.zeros(d), c)[0] == 1
    centre = np.zeros(d)
    centre[1] = np.inf
    assert host_chol(H, centre, cov)[0] == 1


@pytest.mark.parametrize("case", ["gauss", "heavy", "ties", "minus_inf", "small"])
def test_host_summary_matches_numpy(H, case):
    rng = np.random.default_rng(["gauss", "heavy", "ties", "minus_inf", "small"].index(case))
    S = {"small": 7}.get(case, 2000)
    if case == "gauss":
        lw = rng.normal(0, 0.3, S)
    elif case == "heavy":
        lw = 2.0 * rng.standard_t(3, S)
    elif case == "ties":
        lw = np.round(rng.normal(0, 1, S), 1)
    elif case == "minus_inf":
        lw = rng.normal(0, 1, S)
        lw[rng.random(S) < 0.3] = -np.inf
    else:
        lw = rng.normal(0, 1, S)
    u = rng.random()
    st, ess, kh, rs = host_summary(H, lw, u)
    assert st == 0
    assert abs(ess - ess_reference(lw)) <= 1e-12 * ess_reference(lw)
    want = khat_reference(lw)
    if np.isinf(want):
        assert kh == want, (case, kh)
    else:
        assert abs(kh - want) <= 1e-9, (case, kh, want)
    idx, near = resample_reference(lw, u)
    differ = rs != idx
    assert np.all(near[differ] <= 1e-12), case


def test_host_summary_no_weight(H):
    assert host_summary(H, np.full(10, -np.inf), 0.5)[0] == 2


@pytest.mark.parametrize("k_true", [0.3, 0.6, 0.9])
def test_host_khat_finds_the_pareto_shape(H, k_true):
    """Weights w = U^-k (a Pareto tail of shape k) at S = 10^5: k-hat estimates k from the largest 3 sqrt(S) weights."""
    rng = np.random.default_rng(int(10 * k_true))
    lw = -k_true * np.log(rng.random(100000))
    st, ess, kh, _ = host_summary(H, lw, 0.5)
    assert st == 0 and abs(kh - k_true) <= 0.1, (k_true, kh)
    assert abs(kh - khat_reference(lw)) <= 1e-9
