"""Survey-scale Kalman smoother (carma_multi_smooth, MultiSeries.smooth): smoothed values, leave-one-out laws and query
interpolation of every curve of a multi-series in one call.

  * loglik is bitwise MultiSeries.loglik (-inf and NaN rows included); a rejected row gives a NaN curve;
  * mean / var agree with MultiSeries.predict at each curve's own data times, qmean / qvar with predict at backcasts,
    forecasts, data times, duplicates and unsorted times, in caller order;
  * on curves of <= 400 points mean, var, loo_mean and loo_var agree with the dense Gaussian-process conditional;
  * outputs are bitwise the same across curve subsets, batch mates, chunking and with or without queries;
  * a planted outlier has its curve's largest leave-one-out |z|, and the z of clean curves are standard normal.

Tolerances (set from a run on a B200, DESIGN.md "Survey smoother"): the smoother and predict are different recursions of
the same conditional law, and the smoothed variance loses digits to the cancellation c P c - g^T Lambda g, so variances
are compared relative to the prior variance v0 = sigma_y^2."""
import numpy as np
import pytest

from test_gpu_survey_filter import LENGTHS, _explicit, _models, _queries, _ragged_survey, _thetas  # noqa: F401

pytestmark = pytest.mark.gpu

# largest errors measured on a B200 over the seven shapes: means 9e-14 x std(y), variances 3.5e-14 x v0; the tolerances
# leave two orders of magnitude for other data
MEAN_TOL = 1e-11   # x std(y) of the curve
VAR_TOL = 1e-12    # x v0


@pytest.fixture(scope="module")
def C():
    import carma_pack_b200 as c
    if c._lib.device_count() < 1:
        pytest.fail("no CUDA device visible: GPU tests must run on the B200 box")
    return c


def _dense(C, kind, p, q, th, t, y, e, prior):
    """Smoothed mean / var at the data times and the leave-one-out law of y from the dense covariance (without mu)."""
    from carma_pack_b200 import synth
    s2, roots, ma = _explicit(C, kind, p, q, th, prior)
    Kf = synth.carma_variance(s2, roots, ma, lag=np.abs(t[:, None] - t[None, :]))
    K = Kf + np.diag(th[1] * e ** 2)
    Ki = np.linalg.inv(K)
    a = Ki @ (y - th[2])
    return Kf @ a, np.diag(Kf - Kf @ Ki @ Kf), (y - th[2]) - a / np.diag(Ki), 1.0 / np.diag(Ki)


def _close(got, want, scale, tol, what):
    err = np.max(np.abs(got - want)) / scale
    assert err <= tol, "%s: %.3g > %.3g" % (what, err, tol)


@pytest.mark.parametrize("model", range(7))
def test_smooth_matches_loglik_predict_and_dense_gp(C, model):
    m, ts, ys, es = _ragged_survey(C)
    name, kind, p, q, tail = _models(C)[model]
    th = _thetas(ys, tail, seed=model)
    pri = m.default_priors()
    rng = np.random.default_rng(model)
    qs = [_queries(rng, t) for t in ts]
    qs[7] = np.zeros(0)                               # a curve without queries
    qo = np.cumsum([0] + [x.size for x in qs])
    tq = np.concatenate(qs)
    r = m.smooth(kind, p, q, th, tq=tq, q_offsets=qo)
    ll = m.loglik(kind, p, q, th, flags=0 if p == 1 else C.IGNORE_BOUNDS)
    np.testing.assert_array_equal(r.loglik, ll, err_msg=name)          # bitwise, -inf and NaN rows included
    if p == 1:                                        # flags 0: sigma_y < 0 fails the prior bounds
        assert r.loglik[1] == -np.inf
    assert not np.isfinite(r.loglik[4])
    # at the data times: predict with every data time as a query
    pm, pv = m.predict(kind, p, q, th, np.concatenate(ts), m.offsets)
    qm, qv = m.predict(kind, p, q, th, tq, qo)
    off = m.offsets
    for c in range(m.ncurves):
        sl, ql = slice(off[c], off[c + 1]), slice(qo[c], qo[c + 1])
        if r.loglik[c] == -np.inf:                    # rejected by the transform: the whole curve is NaN
            for key in ("mean", "var", "loo_mean", "loo_var"):
                assert np.all(np.isnan(r[key][sl])), (name, c, key)
            assert np.all(np.isnan(r.qmean[ql])) and np.all(np.isnan(r.qvar[ql]))
            continue
        if not np.isfinite(r.loglik[c]):
            continue
        sy, v0 = np.std(ys[c]), th[c, 0] ** 2
        what = "%s curve %d" % (name, c)
        _close(r.mean[sl], pm[sl], sy, MEAN_TOL, what + " mean vs predict")
        _close(r.var[sl], pv[sl], v0, VAR_TOL, what + " var vs predict")
        if qs[c].size:
            _close(r.qmean[ql], qm[ql], sy, MEAN_TOL, what + " qmean vs predict")
            _close(r.qvar[ql], qv[ql], v0, VAR_TOL, what + " qvar vs predict")
        if ts[c].size <= 400:
            t, y, e = m.curve(c)
            dm, dv, dlm, dlv = _dense(C, kind, p, q, th[c], t, y, e, C.Prior(*pri[c]))
            _close(r.mean[sl] - th[c, 2], dm, sy, MEAN_TOL, what + " mean vs dense")
            _close(r.var[sl], dv, v0, VAR_TOL, what + " var vs dense")
            _close(r.loo_mean[sl] - th[c, 2], dlm, sy, MEAN_TOL, what + " loo_mean vs dense")
            _close(r.loo_var[sl], dlv, v0, VAR_TOL, what + " loo_var vs dense")
    m.close()


def test_outputs_are_bitwise_invariant(C, monkeypatch):
    m, ts, ys, es = _ragged_survey(C, seed=9)
    name, kind, p, q, tail = _models(C)[4]
    th = _thetas(ys, tail, seed=4, bad=False)
    rng = np.random.default_rng(3)
    qs = [_queries(rng, t) for t in ts]
    qo = np.cumsum([0] + [x.size for x in qs])
    tq = np.concatenate(qs)
    full = m.smooth(kind, p, q, th, tq=tq, q_offsets=qo)
    keys = ("mean", "var", "loo_mean", "loo_var", "loglik", "qmean", "qvar")
    # without queries
    nq = m.smooth(kind, p, q, th)
    assert "qmean" not in nq and "qvar" not in nq
    for key in keys[:5]:
        np.testing.assert_array_equal(nq[key], full[key], err_msg=key)
    # queries only
    qonly = m.smooth(kind, p, q, th, tq=tq, q_offsets=qo, points=False)
    assert "mean" not in qonly and "loo_var" not in qonly
    for key in keys[4:]:
        np.testing.assert_array_equal(qonly[key], full[key], err_msg="points=False " + key)
    # several chunks
    monkeypatch.setenv("CARMA_MULTI_SMOOTH_BUDGET", "20000")
    ch = m.smooth(kind, p, q, th, tq=tq, q_offsets=qo)
    monkeypatch.delenv("CARMA_MULTI_SMOOTH_BUDGET")
    for key in keys:
        np.testing.assert_array_equal(ch[key], full[key], err_msg="chunked " + key)
    # a subset of the curves, with other batch mates
    k, n = 9, 6
    off = np.cumsum([0] + [t.size for t in ts[k:k + n]])
    part = C.MultiSeries(np.concatenate(ts[k:k + n]), np.concatenate(ys[k:k + n]), np.concatenate(es[k:k + n]), off)
    pqo = np.cumsum([0] + [x.size for x in qs[k:k + n]])
    pr = part.smooth(kind, p, q, th[k:k + n], tq=np.concatenate(qs[k:k + n]), q_offsets=pqo)
    lo, hi = m.offsets[k], m.offsets[k + n]
    for key in keys[:4]:
        np.testing.assert_array_equal(pr[key], full[key][lo:hi], err_msg="subset " + key)
    np.testing.assert_array_equal(pr.loglik, full.loglik[k:k + n])
    np.testing.assert_array_equal(pr.qmean, full.qmean[qo[k]:qo[k + n]])
    np.testing.assert_array_equal(pr.qvar, full.qvar[qo[k]:qo[k + n]])
    # caller order: a permutation of the queries within each curve permutes the answers
    curve_of = np.repeat(np.arange(m.ncurves), np.diff(qo))
    order = np.lexsort((rng.permutation(tq.size), curve_of))
    po = m.smooth(kind, p, q, th, tq=tq[order], q_offsets=qo)
    np.testing.assert_array_equal(po.qmean, full.qmean[order])
    np.testing.assert_array_equal(po.qvar, full.qvar[order])
    part.close()
    m.close()


def test_rejected_rows_leave_their_neighbours_alone(C):
    m, ts, ys, es = _ragged_survey(C, seed=5)
    name, kind, p, q, tail = _models(C)[2]
    clean = _thetas(ys, tail, seed=6, bad=False)
    bad = clean.copy()
    bad[1, 0] = -1.0
    bad[4, 3] = np.nan
    rng = np.random.default_rng(6)
    qs = [_queries(rng, t) for t in ts]
    qo = np.cumsum([0] + [x.size for x in qs])
    tq = np.concatenate(qs)
    a = m.smooth(kind, p, q, clean, tq=tq, q_offsets=qo, flags=0)
    b = m.smooth(kind, p, q, bad, tq=tq, q_offsets=qo, flags=0)
    assert b.loglik[1] == -np.inf and not np.isfinite(b.loglik[4])
    off = m.offsets
    for c in range(m.ncurves):
        sl, ql = slice(off[c], off[c + 1]), slice(qo[c], qo[c + 1])
        for key, s in (("mean", sl), ("var", sl), ("loo_mean", sl), ("loo_var", sl), ("qmean", ql), ("qvar", ql)):
            if c in (1, 4):
                assert np.all(np.isnan(b[key][s])), (c, key)
            else:
                np.testing.assert_array_equal(b[key][s], a[key][s], err_msg="%d %s" % (c, key))
    m.close()


def test_loo_residuals_flag_an_outlier_and_are_standard_normal(C):
    from carma_pack_b200 import synth
    th = synth.carma31_theta()
    nc, ny = 10000, 100
    sim = C.MultiSeries.simulate(nc, ny, C.KIND_CARMA, 3, 1, th, yerr=0.2, dt_min=0.05, dt_max=60.0, seed=41)
    curves = [sim.curve(c) for c in range(nc)]
    sim.close()
    t = np.concatenate([x[0] for x in curves])
    y = np.concatenate([x[1] for x in curves])
    e = np.concatenate([x[2] for x in curves])
    off = np.arange(nc + 1) * ny
    theta = np.tile(th, (nc, 1))
    m = C.MultiSeries(t, y, e, off)
    r = m.smooth(C.KIND_CARMA, 3, 1, theta)
    z = (y - r.loo_mean) / np.sqrt(r.loo_var)
    assert np.all(np.isfinite(z))
    assert abs(z.mean()) < 0.01 and abs(z.std() - 1.0) < 0.01, (z.mean(), z.std())
    m.close()
    # plant a 10 sigma outlier in some curves, each at its own point
    rng = np.random.default_rng(7)
    nbad = 64
    where = rng.integers(0, ny, nbad)
    y2 = y.copy()
    y2[np.arange(nbad) * ny + where] += 10.0 * np.sqrt(r.loo_var[np.arange(nbad) * ny + where])
    m2 = C.MultiSeries(t, y2, e, off)
    r2 = m2.smooth(C.KIND_CARMA, 3, 1, theta)
    z2 = np.abs((y2 - r2.loo_mean) / np.sqrt(r2.loo_var)).reshape(nc, ny)
    np.testing.assert_array_equal(np.argmax(z2[:nbad], axis=1), where)
    m2.close()


def test_argument_checks(C):
    m, ts, ys, es = _ragged_survey(C)
    name, kind, p, q, tail = _models(C)[2]
    th = _thetas(ys, tail, seed=1, bad=False)
    L = C._lib.lib
    qo = np.zeros(m.ncurves + 1, dtype=np.int64)
    qo[5:] = 2
    qo[9] = 1                                         # decreasing
    tq = np.zeros(2)
    out = np.empty(m.offsets[-1])
    rc = L.carma_multi_smooth(m.handle, kind, p, q, None, th.ctypes.data, 1, out.ctypes.data, None, None, None, None,
                              qo.ctypes.data, tq.ctypes.data, None, None)
    assert rc != 0 and b"non-decreasing" in L.carma_last_error()
    qo[9] = 2
    tq[1] = np.nan
    rc = L.carma_multi_smooth(m.handle, kind, p, q, None, th.ctypes.data, 1, out.ctypes.data, None, None, None, None,
                              qo.ctypes.data, tq.ctypes.data, None, None)
    assert rc != 0 and b"non-finite" in L.carma_last_error()
    rc = L.carma_multi_smooth(m.handle, C.KIND_CARMA, 3, 3, None, th.ctypes.data, 1, out.ctypes.data, None, None, None,
                              None, None, None, None, None)
    assert rc != 0 and b"invalid" in L.carma_last_error()
    # every output may be NULL: only the mean requested
    rc = L.carma_multi_smooth(m.handle, kind, p, q, None, th.ctypes.data, 1, out.ctypes.data, None, None, None, None,
                              None, None, None, None)
    assert rc == 0
    np.testing.assert_array_equal(out + np.repeat(th[:, 2], np.diff(m.offsets)), m.smooth(kind, p, q, th).mean)
    m.close()
