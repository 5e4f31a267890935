"""Survey-scale Laplace importance sampling (carma_multi_laplace, MultiSeries.laplace / laplace_sample,
CarmaModel.laplace_sample): draws from N(theta_c, cov_c), their exact log-densities, the weight ESS, the Pareto k-hat
and a systematic resample of every curve in one call.

  * logpost is bitwise MultiSeries.loglik of the draws (-inf rows included);
  * the draws are the documented Philox / Box-Muller / Cholesky rows, rebuilt in numpy, and logq their proposal density;
  * outputs are bitwise the same across batch mates, curve subsets with a matching curve_offset, ndraws prefixes,
    chunking, and CarmaModel(curve).laplace_sample;
  * ess, khat and resample are the numpy references of tests/test_survey_laplace_host.py on the device's weights;
  * each status has its documented cause, and no other curve is affected;
  * the raw draws reproduce theta and cov;
  * at the get_mle fits and hessian covariances of simulated CAR(1) / CAR(2) surveys, k-hat <= 0.7 for most curves, and
    a proposal far too narrow (cov x 0.05) makes it fire;
  * on well-constrained curves the resampled quantiles and the PSD band agree with run_mcmc's.

Ceilings were set from a run on a B200 (DESIGN.md "Survey Laplace importance sampling")."""
import numpy as np
import pytest

from test_gpu_survey_filter import _models, _ragged_survey, _thetas
from test_survey_laplace_host import chol_reference, ess_reference, khat_reference, resample_reference

pytestmark = pytest.mark.gpu

CARMA_ERR_ARG = 1
EPS = np.finfo(float).eps


@pytest.fixture(scope="module")
def C():
    import carma_pack_b200 as c
    if c._lib.device_count() < 1:
        pytest.fail("no CUDA device visible: GPU tests must run on the B200 box")
    return c


def _covs(th, seed, scale=0.01):
    """A positive-definite proposal covariance per curve: (scale |theta| + 1e-3)^2-sized, mildly correlated."""
    rng = np.random.default_rng(seed)
    nc, d = th.shape
    out = np.empty((nc, d, d))
    for c in range(nc):
        s = scale * np.abs(np.nan_to_num(th[c])) + 1e-3
        A = rng.normal(size=(d, d)) * 0.3 + np.eye(d)
        R = A @ A.T
        R /= np.sqrt(np.outer(np.diag(R), np.diag(R)))
        out[c] = R * np.outer(s, s)
    return out


def _philox_rows(O, th, cov, seed, curve, S):
    """The documented draws of one curve in numpy: z from the oracle's Philox and Box-Muller, L by the documented loop,
    rows theta + L z with s accumulated left to right."""
    d = th.size
    L, ld = chol_reference(cov)
    npair = (d + 1) // 2
    z = np.empty((S, 2 * npair))
    for j in range(S):
        for k in range(npair):
            w = O.philox(curve, k, j, 6, seed)
            u0 = ((w[0] >> 5) * 67108864.0 + (w[1] >> 6) + 0.5) * (1.0 / 9007199254740992.0)
            u1 = ((w[2] >> 5) * 67108864.0 + (w[3] >> 6) + 0.5) * (1.0 / 9007199254740992.0)
            r = np.sqrt(-2.0 * np.log(u0))
            z[j, 2 * k], z[j, 2 * k + 1] = r * np.cos(6.283185307179586 * u1), r * np.sin(6.283185307179586 * u1)
    z = z[:, :d]
    rows = np.empty((S, d))
    scale = np.empty((S, d))
    for i in range(d):
        s = np.zeros(S)
        for k in range(i + 1):
            s = s + L[i, k] * z[:, k]
        rows[:, i] = th[i] + s
        scale[:, i] = np.abs(th[i]) + np.abs(L[i, :i + 1] * z[:, :i + 1]).sum(axis=1)
    logq = -0.5 * (z ** 2).sum(axis=1) - ld - 0.5 * d * np.log(2 * np.pi)
    return rows, logq, scale


@pytest.mark.parametrize("model", range(7))
def test_logpost_is_loglik_of_the_draws(C, model):
    m, ts, ys, es = _ragged_survey(C)
    name, kind, p, q, tail = _models(C)[model]
    th = _thetas(ys, tail, seed=model, bad=False)
    S = 64
    flags = 0 if p == 1 else C.IGNORE_BOUNDS   # rows near the model: under flags 0 the prior rejects many of them
    r = m.laplace(kind, p, q, th, _covs(th, model), ndraws=S, seed=11, flags=flags)
    assert r.draws.shape == (m.ncurves, S, th.shape[1]) and r.logpost.shape == r.logq.shape == (m.ncurves, S)
    # NO_WEIGHT exactly where no draw has a finite logpost (curves of two or three points can leave the prior)
    none = np.all(r.logpost == -np.inf, axis=1)
    np.testing.assert_array_equal(r.status, np.where(none, C.LAPLACE_NO_WEIGHT, C.LAPLACE_OK), err_msg=name)
    assert np.mean(r.status == C.LAPLACE_OK) >= 0.8, (name, r.status)
    for j in range(S):
        ll = m.loglik(kind, p, q, np.ascontiguousarray(r.draws[:, j]), flags=flags)
        np.testing.assert_array_equal(r.logpost[:, j], ll, err_msg="%s draw %d" % (name, j))
    np.testing.assert_array_equal(r.log_weights, np.where(np.isfinite(r.logpost), r.logpost - r.logq, -np.inf))
    # a wide proposal under the prior bounds (flags 0, the default): many rows leave the prior, -inf here too
    wide = m.laplace(kind, p, q, th, _covs(th, model, scale=0.5), ndraws=S, seed=12)
    assert np.any(wide.logpost == -np.inf), name
    for j in range(0, S, 7):
        np.testing.assert_array_equal(wide.logpost[:, j],
                                      m.loglik(kind, p, q, np.ascontiguousarray(wide.draws[:, j]), flags=0))
    m.close()


@pytest.mark.parametrize("model", [0, 2, 5])
def test_draws_are_the_documented_rows(C, model):
    from oracle import oracle as O
    O.build()
    m, ts, ys, es = _ragged_survey(C)
    name, kind, p, q, tail = _models(C)[model]
    th = _thetas(ys, tail, seed=model, bad=False)
    cov = _covs(th, model)
    S, seed, off = 40, 2 ** 40 + 3, 1000
    r = m.laplace(kind, p, q, th, cov, ndraws=S, seed=seed, curve_offset=off)
    for c in (0, 3, 12):
        rows, logq, scale = _philox_rows(O, th[c], cov[c], seed, off + c, S)
        assert np.all(np.abs(r.draws[c] - rows) <= 4 * EPS * scale), (name, c)
        np.testing.assert_allclose(r.logq[c], logq, rtol=1e-13, atol=0)
    m.close()


def test_outputs_are_bitwise_invariant(C, monkeypatch):
    import carma_pack_b200 as cp
    m, ts, ys, es = _ragged_survey(C, seed=9)
    keys = ("draws", "logpost", "logq", "resample", "ess", "khat", "status")
    for model in (0, 2, 4):
        name, kind, p, q, tail = _models(C)[model]
        th = _thetas(ys, tail, seed=model, bad=False)
        cov = _covs(th, model)
        S = 200
        full = m.laplace(kind, p, q, th, cov, ndraws=S, seed=5)
        # batch mates: every other curve's row and covariance change
        th2, cov2 = th.copy(), cov.copy()
        th2[1::2, 3:] += 0.05
        cov2[1::2] *= 2.0
        mates = m.laplace(kind, p, q, th2, cov2, ndraws=S, seed=5)
        for key in keys:
            np.testing.assert_array_equal(mates[key][0::2], full[key][0::2], err_msg=key)
        # a prefix of the draws
        pre = m.laplace(kind, p, q, th, cov, ndraws=S // 2, seed=5)
        for key in ("draws", "logpost", "logq"):
            np.testing.assert_array_equal(pre[key], full[key][:, :S // 2], err_msg="prefix " + key)
        # several chunks: three curves per chunk
        d = th.shape[1]
        monkeypatch.setenv("CARMA_MULTI_LAPLACE_BUDGET", str(3 * (8 * S * (d + 3) + 4 * S + 8 * d * d + 32)))
        ch = m.laplace(kind, p, q, th, cov, ndraws=S, seed=5)
        monkeypatch.delenv("CARMA_MULTI_LAPLACE_BUDGET")
        for key in keys:
            np.testing.assert_array_equal(ch[key], full[key], err_msg="chunked " + key)
        # a subset of the curves in a multi-series of their own, with the matching curve_offset
        sub = [7, 8, 9, 10]
        ms = C.MultiSeries(np.concatenate([ts[c] for c in sub]), np.concatenate([ys[c] for c in sub]),
                           np.concatenate([es[c] for c in sub]), np.cumsum([0] + [len(ts[c]) for c in sub]))
        pri = m.default_priors()[sub]
        part = ms.laplace(kind, p, q, th[sub], cov[sub], ndraws=S, seed=5, curve_offset=7, priors=pri)
        ms.close()
        for key in keys:
            np.testing.assert_array_equal(part[key], full[key][sub], err_msg="subset " + key)
        # the single-curve form against a one-curve survey
        for c in (0, 5):
            one = cp.CarmaModel(ts[c], ys[c], es[c], p=p, q=q).laplace_sample(th[c], cov=cov[c], ndraws=S, seed=5)
            m1 = C.MultiSeries(ts[c], ys[c], es[c], [0, len(ts[c])])
            s1 = m1.laplace_sample(p, q, th[c][None], cov=cov[c][None], ndraws=S, seed=5)
            m1.close()
            np.testing.assert_array_equal(one._trace, s1.trace[0], err_msg="CarmaModel %s" % name)
            np.testing.assert_array_equal([one.khat, one.ess, one.status], [s1.khat[0], s1.ess[0], s1.status[0]])
    m.close()


@pytest.mark.parametrize("S", [5, 100, 1000, 6000])
def test_summaries_match_numpy(C, S):
    from oracle import oracle as O
    O.build()
    m, ts, ys, es = _ragged_survey(C, seed=4)
    name, kind, p, q, tail = _models(C)[2]
    th = _thetas(ys, tail, seed=3, bad=False)
    seed, off = 77, 5
    checked = 0
    for scale in (0.01, 0.1):
        r = m.laplace(kind, p, q, th, _covs(th, 3, scale=scale), ndraws=S, seed=seed, curve_offset=off,
                      flags=C.IGNORE_BOUNDS)
        for c in range(m.ncurves):
            if r.status[c] != C.LAPLACE_OK:
                continue
            lw = r.log_weights[c]
            assert abs(r.ess[c] - ess_reference(lw)) <= 1e-12 * ess_reference(lw), (S, c)
            want = khat_reference(lw)
            if np.isinf(want):
                assert r.khat[c] == want, (S, c, r.khat[c])
            else:
                assert abs(r.khat[c] - want) <= 1e-9, (S, c, r.khat[c], want)
            w = O.philox(off + c, 0, 0, 7, seed)
            u = ((w[0] >> 5) * 67108864.0 + (w[1] >> 6) + 0.5) * (1.0 / 9007199254740992.0)
            idx, near = resample_reference(lw, u)
            differ = r.resample[c] != idx
            if differ.any():
                assert near is not None and np.all(near[differ] <= 1e-12), (S, c)
            checked += 1
    assert checked >= 20, checked
    m.close()


def test_status_paths(C):
    m, ts, ys, es = _ragged_survey(C, seed=5)
    name, kind, p, q, tail = _models(C)[2]
    th = _thetas(ys, tail, seed=1, bad=False)
    cov = _covs(th, 1)
    S = 100
    base = m.laplace(kind, p, q, th, cov, ndraws=S, seed=3)
    th2, cov2 = th.copy(), cov.copy()
    cov2[2, 1, 0] = np.nan                     # NaN in the lower triangle
    cov2[5, 3, 3] = -1.0                       # not positive definite
    th2[8, 2] = np.inf                         # a non-finite centre
    th2[11, 0] = -10.0 * abs(th2[11, 0])       # centre outside the prior (sigma_y < 0) with a tiny cov: NO_WEIGHT
    cov2[11] *= 1e-12
    r = m.laplace(kind, p, q, th2, cov2, ndraws=S, seed=3)
    for c in (2, 5, 8):
        assert r.status[c] == C.LAPLACE_BAD_COV, c
        assert np.all(np.isnan(r.draws[c])) and np.all(np.isnan(r.logpost[c])) and np.all(np.isnan(r.logq[c]))
        assert np.isnan(r.khat[c]) and r.ess[c] == 0 and np.all(r.resample[c] == -1)
        assert np.all(np.isnan(r.log_weights[c]))
    assert r.status[11] == C.LAPLACE_NO_WEIGHT
    assert np.all(np.isfinite(r.draws[11])) and np.all(np.isfinite(r.logq[11])) and np.all(r.logpost[11] == -np.inf)
    assert np.isnan(r.khat[11]) and r.ess[11] == 0 and np.all(r.resample[11] == -1)
    rest = np.setdiff1d(np.arange(m.ncurves), [2, 5, 8, 11])
    for key in ("draws", "logpost", "logq", "resample", "ess", "khat", "status"):
        np.testing.assert_array_equal(r[key][rest], base[key][rest], err_msg=key)
    # the upper triangle is never read
    cov3 = cov.copy()
    cov3[4, 0, 3] = np.nan
    np.testing.assert_array_equal(m.laplace(kind, p, q, th, cov3, ndraws=S, seed=3).draws, base.draws)
    # curve_offset + ncurves past 2^32, before any launch
    rc = C._lib.lib.carma_multi_laplace(m.handle, kind, p, q, None, th.ctypes.data, cov.ctypes.data, 0, S, 3,
                                        2 ** 32 - m.ncurves + 1, None, None, None, None, None, None, None)
    assert rc == CARMA_ERR_ARG and b"curve_offset" in C._lib.lib.carma_last_error()
    # laplace_sample: NaN trace rows for the non-OK curves
    ls = m.laplace_sample(p, q, th2, cov=cov2, ndraws=S, seed=3)
    for c in (2, 5, 8, 11):
        assert np.all(np.isnan(ls.trace[c])) and np.all(np.isnan(ls.logpost[c]))
    okr = rest[ls.status[rest] == C.LAPLACE_OK]
    assert okr.size >= 5 and np.all(np.isfinite(ls.trace[okr]))
    m.close()


def test_draws_reproduce_theta_and_cov(C):
    m, ts, ys, es = _ragged_survey(C, seed=6)
    name, kind, p, q, tail = _models(C)[2]
    th = _thetas(ys, tail, seed=2, bad=False)
    cov = _covs(th, 2, scale=0.05)
    S = 100000
    r = m.laplace(kind, p, q, th, cov, ndraws=S, seed=8)
    for c in (0, 6, 12):
        x = r.draws[c]
        sd = np.sqrt(np.diag(cov[c]))
        z = (x.mean(axis=0) - th[c]) / (sd / np.sqrt(S))
        assert np.all(np.abs(z) < 5.0), (c, z)
        corr_err = (np.cov(x.T) - cov[c]) / np.outer(sd, sd)
        assert np.abs(corr_err).max() < 6.0 * np.sqrt(2.0 / S), (c, np.abs(corr_err).max())
    m.close()


CALIBRATION = [   # (name, p, q, theta_true, ncurves, ny), the calibration cases of test_gpu_survey_hessian.py
    ("car1", 1, 0, [1.0, 1.0, 0.0, np.log(1.0 / 3.0)], 3000, 1000),
    ("car2", 2, 0, None, 3000, 600),
]
# the least fraction of curves with k-hat <= 0.7 at the fits, 1000 draws each.  Measured on a B200: CAR(1) 0.846 (median
# k-hat 0.56, median weight ESS 697), CAR(2) 0.961 (median 0.45, ESS 814); cov x 0.05 fires on 0.955 and 0.975
KHAT_OK_FLOOR = {"car1": 0.8, "car2": 0.9}


def _truth(case):
    from carma_pack_b200 import synth
    name, p, q, truth, nc, ny = CALIBRATION[case]
    if truth is None:
        truth = [1.0, 1.0, 0.0] + list(synth.roots_to_logquad(np.array([-0.1 + 0.6j, -0.1 - 0.6j])))
    return name, p, q, np.array(truth), nc, ny


@pytest.mark.parametrize("case", range(len(CALIBRATION)))
def test_khat_at_the_fits(C, case):
    name, p, q, truth, nc, ny = _truth(case)
    kind = C.KIND_CAR1 if p == 1 else C.KIND_CARP
    m = C.MultiSeries.simulate(nc, ny, kind, p, q, truth, yerr=0.05, dt_min=0.05, dt_max=20.0, seed=31 + case)
    fit = m.get_mle(p, q, ntrials=8, seed=7)
    h = m.hessian(kind, p, q, fit.x)
    ok = h.status == C.HESS_OK
    ls = m.laplace_sample(p, q, fit.x, ndraws=1000, seed=1)
    assert np.all(ls.status[~ok] == C.LAPLACE_BAD_COV) and np.all(ls.status[ok] == C.LAPLACE_OK), name
    good = np.mean(ls.khat[ok] <= 0.7)
    assert good >= KHAT_OK_FLOOR[name], (name, good, np.quantile(ls.khat[ok], [0.5, 0.9, 0.99]))
    narrow = m.laplace(kind, p, q, fit.x, np.where(ok[:, None, None], h.cov, np.nan) * 0.05, ndraws=1000, seed=1)
    fires = np.mean(narrow.khat[ok] > 0.7)
    assert fires >= 0.9, (name, fires, np.quantile(narrow.khat[ok], [0.01, 0.1, 0.5]))
    m.close()


def test_resampled_posterior_agrees_with_mcmc(C):
    """CAR(1) curves of 1000 points: well constrained, so the Laplace proposal covers the posterior."""
    name, p, q, truth, nc, ny = _truth(0)
    nc = 50
    m = C.MultiSeries.simulate(nc, ny, C.KIND_CAR1, p, q, truth, yerr=0.05, dt_min=0.05, dt_max=20.0, seed=41)
    fit = m.get_mle(p, q, ntrials=8, seed=7)
    ls = m.laplace_sample(p, q, fit.x, ndraws=4000, seed=2)
    mc = m.run_mcmc(p, q, 4000, seed=3)
    keep = (ls.status == C.LAPLACE_OK) & (ls.khat <= 0.7)
    assert keep.mean() >= KHAT_OK_FLOOR["car1"], keep.mean()
    cols = [0, 2, 3]
    for arr in (ls.trace, mc.trace):
        assert arr.shape[0] == nc
    qs = [16, 50, 84]
    a = np.percentile(ls.trace[keep][:, :, cols], qs, axis=1)
    b = np.percentile(mc.trace[keep][:, :, cols], qs, axis=1)
    sd = mc.trace[keep][:, :, cols].std(axis=1)
    dev = np.abs(a - b) / sd[None]
    assert np.median(dev) <= 0.1 and dev.max() <= 0.5, (np.median(dev), dev.max())
    lo_l, hi_l, mid_l, f = ls.psd_credible_band(68.0)
    lo_m, hi_m, mid_m, _ = mc.psd_credible_band(68.0)
    width = np.log(hi_m[keep]) - np.log(lo_m[keep])
    for x, y in ((lo_l, lo_m), (hi_l, hi_m), (mid_l, mid_m)):
        err = np.abs(np.log(x[keep]) - np.log(y[keep])) / width
        assert np.median(err) <= 0.1 and err.max() <= 0.5, (np.median(err), err.max())
    with pytest.raises(ValueError, match=r"\.ess"):
        ls.effective_samples("mu")
    m.close()
