"""The recursion the CUDA kernels run, compiled for the HOST and compared with the oracle on the CPU.

csrc/theta_transform.cuh, kalman_real.cuh and fast_math.cuh are __host__ __device__ code; tests/host_check/hostcheck.cu
instantiates their host side (test infrastructure, not part of libcarma_b200.so).  What this pins without a GPU:
the real-half state with D = P - V, the sum/difference basis of real root pairs with the (ch, sh) "hyperbolic
rotation", the pre-scaled range reductions of exp / sin / cos, the branch-free mantissa-product form of sum(log var)
and its exact slow path.  The GPU parity tests (tests/test_gpu_parity.py) check the same code as compiled for sm_100a."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import build_native
from carma_pack_b200 import synth
from oracle import oracle as O
from parity_util import assert_logpost_parity, ulp_shift

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "host_check", "hostcheck.cu")
LIB = os.path.join(HERE, "host_check", "libhostcheck.so")
CSRC = os.path.join(os.path.dirname(HERE), "carma_pack_b200", "csrc")
_dp = ctypes.POINTER(ctypes.c_double)


def _build():
    deps = [SRC] + [os.path.join(CSRC, f) for f in ("kalman_real.cuh", "fast_math.cuh", "theta_transform.cuh", "device_math.cuh")]
    if os.path.exists(LIB) and all(os.path.getmtime(LIB) >= os.path.getmtime(d) for d in deps):
        return
    subprocess.check_call([build_native.NVCC, "-O2", "-std=c++17", "-Xcompiler", "-fPIC", "-shared", "--expt-relaxed-constexpr",
                           "-Wno-deprecated-gpu-targets", "-o", LIB, SRC], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)


@pytest.fixture(scope="module")
def H():
    _build()
    L = ctypes.CDLL(LIB)
    L.hostcheck_loglik.restype = ctypes.c_int
    return L


def host_loglik(L, kind, p, q, t, y, e, theta, prior, flags=0, force_generic=0, force_slow=0):
    t = np.ascontiguousarray(t, float); y = np.ascontiguousarray(y, float); e = np.ascontiguousarray(e, float)
    th = np.ascontiguousarray(np.atleast_2d(theta), float)
    out = np.empty(th.shape[0])
    rc = L.hostcheck_loglik(kind, p, q, ctypes.c_uint(flags), ctypes.byref(prior), t.ctypes.data_as(_dp), y.ctypes.data_as(_dp),
                            e.ctypes.data_as(_dp), ctypes.c_size_t(t.size), th.ctypes.data_as(_dp), ctypes.c_size_t(th.shape[0]),
                            out.ctypes.data_as(_dp), force_generic, force_slow)
    assert rc == 0
    return out


def parity(got, want, want_ld, max_noisy_frac=0.01, what="", ulp_eval=None):
    fin = np.isfinite(want)
    assert np.array_equal(np.isnan(want), np.isnan(got))
    assert_logpost_parity(got, want, want_ld, max_illcond_frac=max_noisy_frac, what="host: " + what, ulp_eval=ulp_eval)
    return np.abs(got[fin] - want[fin]) / np.maximum(np.abs(want[fin]), 1.0)


def overdamped(th, p, rng, frac=0.5):
    """Turn quadratic factors of some rows into two REAL roots (discriminant > 0): q2^2 > 4 q1."""
    th = th.copy()
    for s in range(p // 2):
        pick = rng.uniform(size=th.shape[0]) < frac
        q1 = np.exp(th[pick, 3 + 2 * s])
        th[pick, 4 + 2 * s] = np.log(np.sqrt(4.0 * q1) * rng.uniform(1.05, 6.0, pick.sum()))
    return th


def test_config2_shape_against_oracle(H):
    t, y, e = synth.readme_series(270, 270)
    th = synth.theta_batch(3000, t, y, seed=5)
    pr = O.default_prior(t, y)
    want = O.logdensity(O.KIND_CARMA, 5, 3, t, y, e, th, prior=pr)
    want_ld = O.logdensity(O.KIND_CARMA, 5, 3, t, y, e, th, prior=pr, long_double=True)
    got = host_loglik(H, O.KIND_CARMA, 5, 3, t, y, e, th, pr)
    err = parity(got, want, want_ld, max_noisy_frac=0.002, what="config-2 shape CARMA(5,3)",
                 ulp_eval=lambda rows, k: O.logdensity(O.KIND_CARMA, 5, 3, t, y, e, ulp_shift(th[rows], k), prior=pr))
    assert np.median(err) < 1e-13
    # warp-composition independence: the generic loop gives the same bits as the all-conjugate loop
    gen = host_loglik(H, O.KIND_CARMA, 5, 3, t, y, e, th, pr, force_generic=1)
    assert np.array_equal(np.nan_to_num(gen, nan=1.5, neginf=2.5), np.nan_to_num(got, nan=1.5, neginf=2.5))
    # the software-pipelined loop (single-ensemble PT runs) performs the same operations: same bits
    pip = host_loglik(H, O.KIND_CARMA, 5, 3, t, y, e, th, pr, force_generic=2)
    assert np.array_equal(np.nan_to_num(pip, nan=1.5, neginf=2.5), np.nan_to_num(got, nan=1.5, neginf=2.5))


@pytest.mark.parametrize("p", [1, 2, 3, 4, 5, 6, 7])
def test_all_orders_with_real_root_pairs(H, p):
    rng = np.random.default_rng(100 + p)
    t, y, e = synth.readme_series(150, 11)
    pr = O.default_prior(t, y)
    for q in range(0, p):
        if p == 1:
            kind = O.KIND_CAR1
            th = np.column_stack([np.sqrt(np.var(y)) * rng.uniform(0.5, 2, 64), rng.uniform(0.6, 1.9, 64), np.mean(y) + 0.1 * rng.standard_normal(64),
                                  rng.uniform(np.log(pr.min_freq * 1.1), np.log(pr.max_freq * 0.9), 64)])
        else:
            kind = O.KIND_CARMA if q else O.KIND_CARP
            th = overdamped(synth.prior_draws(96, p, q, t, y, rng), p, rng)
        want = O.logdensity(kind, p, q, t, y, e, th, prior=pr, ignore_prior=(p > 1))
        want_ld = O.logdensity(kind, p, q, t, y, e, th, prior=pr, ignore_prior=(p > 1), long_double=True)
        got = host_loglik(H, kind, p, q, t, y, e, th, pr, flags=(1 if p > 1 else 0))
        parity(got, want, want_ld, max_noisy_frac=0.15, what="p=%d q=%d with real pairs" % (p, q),
               ulp_eval=lambda rows, k: O.logdensity(kind, p, q, t, y, e, ulp_shift(th[rows], k), prior=pr, ignore_prior=(p > 1)))
        slow = host_loglik(H, kind, p, q, t, y, e, th, pr, flags=(1 if p > 1 else 0), force_slow=1)
        fin = np.isfinite(got)
        assert np.allclose(slow[fin], got[fin], rtol=2e-12, atol=1e-10)


def test_zcarma_and_zcar(H):
    rng = np.random.default_rng(3)
    t, y, e = synth.readme_series(200, 5)
    pr = O.default_prior(t, y)
    th = np.column_stack([synth.prior_draws(128, 5, 0, t, y, rng), rng.uniform(-3, 3, 128)])
    want = O.logdensity(O.KIND_ZCARMA, 5, 0, t, y, e, th, prior=pr)
    want_ld = O.logdensity(O.KIND_ZCARMA, 5, 0, t, y, e, th, prior=pr, long_double=True)
    got = host_loglik(H, O.KIND_ZCARMA, 5, 0, t, y, e, th, pr)
    parity(got, want, want_ld, max_noisy_frac=0.05, what="ZCARMA(5)")
    z = host_loglik(H, O.KIND_ZCAR, 5, 0, t, y, e, th[:, :8], pr)
    c = host_loglik(H, O.KIND_CARP, 5, 0, t, y, e, th[:, :8], pr)
    assert np.array_equal(np.nan_to_num(z, neginf=1.0), np.nan_to_num(c, neginf=1.0))


def test_long_gaps_and_extreme_variances_take_the_exact_path(H):
    """Season gaps make e^{w dt} underflow (exponent clamp instead of a branch); variances outside the normal
    range raise the sticky flag and the evaluation is redone with one log() per point."""
    rng = np.random.default_rng(8)
    t = np.cumsum(np.concatenate([rng.uniform(0.5, 1.5, 60), [4000.0], rng.uniform(0.5, 1.5, 60), [30000.0], rng.uniform(0.5, 1.5, 40)]))
    y = 3.0 * rng.standard_normal(t.size)
    e = np.full(t.size, 0.3)
    pr = O.default_prior(t, y)
    th = overdamped(synth.prior_draws(200, 4, 1, t, y, rng), 4, rng)
    want = O.logdensity(O.KIND_CARMA, 4, 1, t, y, e, th, prior=pr, ignore_prior=True)
    want_ld = O.logdensity(O.KIND_CARMA, 4, 1, t, y, e, th, prior=pr, ignore_prior=True, long_double=True)
    got = host_loglik(H, O.KIND_CARMA, 4, 1, t, y, e, th, pr, flags=1)
    parity(got, want, want_ld, max_noisy_frac=0.1, what="season gaps CARMA(4,1)",
           ulp_eval=lambda rows, k: O.logdensity(O.KIND_CARMA, 4, 1, t, y, e, ulp_shift(th[rows], k), prior=pr, ignore_prior=True))
    # absurd scales: var ~ 1e-320 (subnormal) and ~1e+305
    for s_y, s_e in ((1e-165, 1e-162), (1e152, 1e150)):
        th2 = th[:20].copy()
        th2[:, 0] = s_y
        e2 = np.full(t.size, s_e)
        want = O.logdensity(O.KIND_CARMA, 4, 1, t, y, e2, th2, prior=pr, ignore_prior=True)
        got = host_loglik(H, O.KIND_CARMA, 4, 1, t, y, e2, th2, pr, flags=1)
        assert np.array_equal(np.isfinite(want), np.isfinite(got)) and np.array_equal(np.isnan(want), np.isnan(got))
        fin = np.isfinite(want)
        assert np.allclose(got[fin], want[fin], rtol=1e-9)


def test_loop_transcendentals(H):
    """exp_scaled / rot_scaled / rcp_fast against long double: the error budget of one transition factor."""
    rng = np.random.default_rng(0)
    n = 40000
    lnat = -np.exp(rng.uniform(np.log(1e-6), np.log(50.0), n))          # natural rates
    dt = np.exp(rng.uniform(np.log(1e-2), np.log(30.0), n))
    l_exp = lnat * (64.0 / np.log(2.0))
    outs = [np.empty(n) for _ in range(6)]
    H.hostcheck_fastmath(l_exp.ctypes.data_as(_dp), dt.ctypes.data_as(_dp), ctypes.c_size_t(n), *[o.ctypes.data_as(_dp) for o in outs])
    ex, _, _, s_r, c_r, _ = outs
    x = l_exp.astype(np.longdouble) * dt.astype(np.longdouble) * (np.log(np.longdouble(2)) / 64)
    want = np.exp(x)
    ok = x > -700
    rel = np.abs(ex[ok] - want[ok]) / want[ok]
    assert rel.max() < 4e-16, rel.max()
    assert np.all(ex[~ok] < 1e-300) and np.all(ex >= 0)
    rho = want
    assert np.abs(c_r - (1 + rho) / 2).max() < 3e-16 and np.abs(s_r - (1 - rho) / 2).max() < 3e-16
    # phases: l in units of pi/64 per unit time
    lp = -np.exp(rng.uniform(np.log(1e-3), np.log(1e7), n))
    outs = [np.empty(n) for _ in range(6)]
    H.hostcheck_fastmath(lp.ctypes.data_as(_dp), dt.ctypes.data_as(_dp), ctypes.c_size_t(n), *[o.ctypes.data_as(_dp) for o in outs])
    _, s_c, c_c, _, _, rc = outs
    assert not np.isnan(s_c).any()       # NaN marks a bit difference between the ALLC and the generic variant
    # exact argument reduction in rational arithmetic: (l dt) mod 128 table steps, then long double
    from fractions import Fraction
    pick = rng.choice(n, 4000, replace=False)
    red = np.array([float(((Fraction(float(lp[i])) * Fraction(float(dt[i]))) % 128)) for i in pick], dtype=np.longdouble)
    lo = np.array([float((Fraction(float(lp[i])) * Fraction(float(dt[i]))) % 128 - Fraction(float(red[k]))) for k, i in enumerate(pick)],
                  dtype=np.longdouble)
    ang = (red + lo) * np.longdouble(np.pi) / 64 + (red + lo) * np.longdouble(1.2246467991473532e-16) / 64   # pi = hi + lo
    assert np.abs(s_c[pick] - np.sin(ang)).max() < 4e-16 and np.abs(c_c[pick] - np.cos(ang)).max() < 4e-16
    assert np.abs(rc * lp - 1.0).max() < 5e-16
