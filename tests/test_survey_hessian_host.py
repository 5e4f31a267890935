"""CPU-side checks of carma_multi_hessian / MultiSeries.hessian.

  * the entry point rejects a non-finite rel_step, an invalid (kind, p, q) and a null handle or theta with CARMA_ERR_ARG
    and a message naming it, before any CUDA call; the binding is exported and declared;
  * MultiSeries.hessian checks its arguments before it uses the handle;
  * the stencil rows and the assembly (hessian.cuh, compiled here for the host by tests/host_check/hesscheck.cu) are
    numpy's: rows bit for bit, gradient and Hessian from the CPU oracle's stencil values as numpy assembles them, the
    covariance np.linalg.inv(-H); and each status path gives the documented NaNs."""
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
SRC = os.path.join(HERE, "host_check", "hesscheck.cu")
LIB = os.path.join(HERE, "host_check", "libhesscheck.so")
CSRC = os.path.join(os.path.dirname(HERE), "carma_pack_b200", "csrc")
_dp = ctypes.POINTER(ctypes.c_double)


def test_survey_hessian_rejects_bad_arguments_before_cuda():
    import carma_pack_b200 as C
    L = C._lib.lib
    th = np.zeros(7)
    out = np.zeros(64)

    def call(m=None, kind=C.KIND_CARMA, p=3, q=1, theta=th.ctypes.data, rel_step=0.0):
        return L.carma_multi_hessian(m, kind, p, q, None, theta, 0, rel_step, out.ctypes.data, None, None, None, None)

    for step in (np.nan, np.inf, -np.inf):
        assert call(rel_step=step) == CARMA_ERR_ARG
        assert b"carma_multi_hessian" in L.carma_last_error() and b"rel_step" in L.carma_last_error()
    for kind, p, q in ((C.KIND_CARMA, 3, 3), (C.KIND_CARMA, 0, 0), (C.KIND_CARMA, 8, 1), (9, 2, 0)):
        assert call(kind=kind, p=p, q=q) == CARMA_ERR_ARG
        assert b"carma_multi_hessian" in L.carma_last_error() and b"invalid" in L.carma_last_error()
    assert call() == CARMA_ERR_ARG
    assert b"carma_multi_hessian" in L.carma_last_error() and b"null" in L.carma_last_error()
    fake = ctypes.c_void_p(1)   # never dereferenced: theta is checked first
    assert call(m=fake, theta=None) == CARMA_ERR_ARG
    assert b"null" in L.carma_last_error()


def test_survey_hessian_binding_is_declared():
    import carma_pack_b200 as C
    assert "carma_multi_hessian" in C._lib.EXPORTED_SYMBOLS
    at = C._lib.lib.carma_multi_hessian.argtypes
    assert at is not None and len(at) == 13 and at[7] is ctypes.c_double
    assert callable(C.MultiSeries.hessian) and callable(C.CarmaModel.hessian)
    assert (C.HESS_OK, C.HESS_REJECTED, C.HESS_NONFINITE, C.HESS_NOT_NEGDEF) == (0, 1, 2, 3)
    assert C.HESS_REL_STEP == 2.0 ** -13
    hdr = open(os.path.join(os.path.dirname(HERE), "include", "carma_b200.h")).read()
    assert "#define CARMA_HESS_DEFAULT_REL_STEP 1.220703125e-4" in hdr and 1.220703125e-4 == 2.0 ** -13


def test_hessian_argument_errors_raise_value_error():
    """The shape checks run before the handle is used, so an object without one shows them."""
    import carma_pack_b200 as C
    fake = object.__new__(C.MultiSeries)
    fake.ncurves = 2
    fake.offsets = np.array([0, 3, 6], dtype=np.int64)
    fake.handle = None
    d = C._lib.model_dim(C.KIND_CARMA, 3, 1)
    th = np.ones((2, d))
    with pytest.raises(ValueError, match="theta"):
        fake.hessian(C.KIND_CARMA, 3, 1, np.zeros((3, d)))
    with pytest.raises(ValueError, match="theta"):
        fake.hessian(C.KIND_CARMA, 3, 1, np.zeros((2, d + 1)))
    with pytest.raises(ValueError, match="priors"):
        fake.hessian(C.KIND_CARMA, 3, 1, th, priors=np.zeros(3, dtype=C._lib.PRIOR_DTYPE))
    for step in (np.nan, np.inf):
        with pytest.raises(ValueError, match="rel_step"):
            fake.hessian(C.KIND_CARMA, 3, 1, th, rel_step=step)


def test_hessian_steps():
    import carma_pack_b200 as C
    th = np.array([[0.7, 1.05, 3.0, -2.0, 0.5], [2.5, 0.95, -1.0, 0.1, 0.2]])
    h = C._lib.hessian_steps(th)
    np.testing.assert_array_equal(h[:, 0], th[:, 0] * 2.0 ** -13)
    np.testing.assert_array_equal(h[:, 1], th[:, 1] * 2.0 ** -13)
    np.testing.assert_array_equal(h[:, 2], th[:, 0] * 2.0 ** -13)
    np.testing.assert_array_equal(h[:, 3:], np.full((2, 2), 2.0 ** -13))


# ---- the stencil and the assembly on the host ---------------------------------------------------------------------

@pytest.fixture(scope="module")
def H():
    deps = [SRC] + [os.path.join(CSRC, f) for f in ("hessian.cuh", "theta_transform.cuh", "fast_math.cuh", "device_math.cuh")]
    if not (os.path.exists(LIB) and all(os.path.getmtime(LIB) >= os.path.getmtime(d) for d in deps)):
        subprocess.check_call([build_native.NVCC, "-O2", "-std=c++17", "-Xcompiler", "-fPIC", "-shared",
                               "--expt-relaxed-constexpr", "-Wno-deprecated-gpu-targets", "-o", LIB, SRC],
                              stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    L = ctypes.CDLL(LIB)
    L.hess_rows.argtypes = [ctypes.c_int, _dp, ctypes.c_double, _dp]
    L.hess_assemble_host.argtypes = [ctypes.c_int, _dp, _dp, _dp, _dp, _dp]
    return L


def stencil_rows(theta, rel_step=2.0 ** -13):
    """The documented stencil of carma_multi_hessian in numpy: centre, +h_i e_i, -h_i e_i, then for i < j the pair
    +h_i e_i + h_j e_j, -h_i e_i - h_j e_j."""
    import carma_pack_b200 as C
    th = np.asarray(theta, dtype=np.float64)
    d = th.size
    h = C._lib.hessian_steps(th, rel_step)[0]
    rows = [th.copy()]
    for sgn in (1.0, -1.0):
        for i in range(d):
            r = th.copy()
            r[i] = th[i] + h[i] if sgn > 0 else th[i] - h[i]
            rows.append(r)
    for i in range(d):
        for j in range(i + 1, d):
            rp, rm = th.copy(), th.copy()
            rp[i], rp[j] = th[i] + h[i], th[j] + h[j]
            rm[i], rm[j] = th[i] - h[i], th[j] - h[j]
            rows += [rp, rm]
    return np.array(rows), h


def assemble(f, h):
    """The documented assembly in numpy, in the header's operation order."""
    d = h.size
    f0, fp, fm = f[0], f[1:1 + d], f[1 + d:1 + 2 * d]
    g = (fp - fm) / (2.0 * h)
    Hm = np.empty((d, d))
    for i in range(d):
        Hm[i, i] = (fp[i] - 2.0 * f0 + fm[i]) / (h[i] * h[i])
    r = 0
    for i in range(d):
        for j in range(i + 1, d):
            num = f[1 + 2 * d + 2 * r] - fp[i] - fp[j] + 2.0 * f0 - fm[i] - fm[j] + f[2 + 2 * d + 2 * r]
            Hm[i, j] = Hm[j, i] = num / (2.0 * h[i] * h[j])
            r += 1
    return g, Hm


def host_assemble(L, f, h):
    d = h.size
    f, h = np.ascontiguousarray(f, float), np.ascontiguousarray(h, float)
    g, Hm, cov = np.empty(d), np.empty((d, d)), np.empty((d, d))
    st = L.hess_assemble_host(d, f.ctypes.data_as(_dp), h.ctypes.data_as(_dp), g.ctypes.data_as(_dp),
                              Hm.ctypes.data_as(_dp), cov.ctypes.data_as(_dp))
    return st, g, Hm, cov


def _logquad(roots):
    return list(synth.roots_to_logquad(roots))


HOST_MODELS = [
    ("car1", O.KIND_CAR1, 1, 0, [np.log(0.3)]),
    ("carma31", O.KIND_CARMA, 3, 1, _logquad([-0.05 + 0.3j, -0.05 - 0.3j, -0.4]) + [np.log(2.0)]),
    ("carma53", O.KIND_CARMA, 5, 3, _logquad([-0.05 + 0.3j, -0.05 - 0.3j, -0.2, -0.9, -0.4]) +
     _logquad([-1.5 + 0.5j, -1.5 - 0.5j, -3.0])),
]


@pytest.mark.parametrize("d", [4, 7, 16])
def test_host_stencil_rows_are_numpys_bitwise(H, d):
    rng = np.random.default_rng(d)
    th = np.concatenate([[rng.uniform(0.1, 3.0), rng.uniform(0.9, 1.1), rng.normal(0, 10)], rng.normal(0, 2, d - 3)])
    for rel in (2.0 ** -13, 1e-3):
        want, _ = stencil_rows(th, rel)
        assert want.shape == (d * d + d + 1, d)
        got = np.empty_like(want)
        assert H.hess_rows(d, th.ctypes.data_as(_dp), rel, got.ctypes.data_as(_dp)) == 0
        np.testing.assert_array_equal(got, want)


@pytest.mark.parametrize("model", range(len(HOST_MODELS)))
def test_host_assembly_matches_numpy_on_oracle_values(H, model):
    name, kind, p, q, tail = HOST_MODELS[model]
    rng = np.random.default_rng(70 + model)
    ar, ma, s2 = synth.carma31_truth()
    ny = 300
    t = np.cumsum(rng.uniform(0.2, 3.0, ny))
    y = 2.0 + synth.carma_process(t, s2, ar, ma, rng) + 0.2 * rng.standard_normal(ny)
    e = rng.uniform(0.1, 0.3, ny)
    theta = np.array([np.std(y), 1.0, np.mean(y)] + list(tail))
    prior = O.default_prior(t, y)
    rows, h = stencil_rows(theta)
    f = O.logdensity(kind, p, q, t, y, e, rows, prior=prior, ignore_prior=p > 1, long_double=True)
    assert np.all(np.isfinite(f)), name
    st, g, Hm, cov = host_assemble(H, f, h)
    wg, wH = assemble(f, h)
    # same operations in the same order on the same doubles; only contraction could differ
    scale = np.abs(wH).max()
    assert np.abs(g - wg).max() <= 1e-13 * np.abs(wg).max(), name
    assert np.abs(Hm - wH).max() <= 1e-13 * scale, name
    np.testing.assert_array_equal(Hm, Hm.T)
    if st == 0:
        inv = np.linalg.inv(-wH)
        cond = np.linalg.cond(wH)
        assert np.abs(cov - inv).max() <= 1e-14 * cond * np.abs(inv).max(), (name, cond)
        np.testing.assert_array_equal(cov, cov.T)
    else:
        assert st == 3 and np.all(np.isnan(cov)), (name, st)
        assert np.linalg.eigvalsh(-wH).min() <= 0.0


def test_host_status_paths(H):
    d = 4
    rng = np.random.default_rng(5)
    A = rng.normal(size=(d, d))
    A = A @ A.T + d * np.eye(d)                   # positive definite
    centre = np.array([1.0, 1.0, 0.0, 0.0])      # steps 1e-3 on every coordinate
    rows, h = stencil_rows(centre, 1e-3)
    dx = rows - centre
    quad = lambda s: -0.5 * s * np.einsum("ki,ij,kj->k", dx, A, dx) + dx @ np.arange(1.0, d + 1)   # noqa: E731
    # concave quadratic: OK, exact second differences up to roundoff, cov = A^-1
    st, g, Hm, cov = host_assemble(H, quad(1.0), h)
    assert st == 0
    np.testing.assert_allclose(Hm, -A, rtol=0, atol=1e-6 * np.abs(A).max())
    np.testing.assert_allclose(cov, np.linalg.inv(A), rtol=0, atol=1e-6 * np.abs(np.linalg.inv(A)).max())
    # convex: NOT_NEGDEF, g and H valid, cov NaN
    st, g, Hm, cov = host_assemble(H, quad(-1.0), h)
    assert st == 3 and np.all(np.isfinite(g)) and np.all(np.isfinite(Hm)) and np.all(np.isnan(cov))
    np.testing.assert_allclose(Hm, A, rtol=0, atol=1e-6 * np.abs(A).max())
    # centre -inf: REJECTED
    f = quad(1.0)
    f[0] = -np.inf
    st, g, Hm, cov = host_assemble(H, f, h)
    assert st == 1 and np.all(np.isnan(g)) and np.all(np.isnan(Hm)) and np.all(np.isnan(cov))
    # a non-finite stencil value, or a zero step: NONFINITE
    for k, v in ((3, -np.inf), (17, np.nan), (20, np.inf)):
        f = quad(1.0)
        f[k] = v
        st, g, Hm, cov = host_assemble(H, f, h)
        assert st == 2 and np.all(np.isnan(g)) and np.all(np.isnan(Hm)) and np.all(np.isnan(cov)), k
    hz = h.copy()
    hz[0] = 0.0
    assert host_assemble(H, quad(1.0), hz)[0] == 2
