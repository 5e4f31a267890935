"""Survey-scale conditional simulation (carma_multi_simulate, MultiSeries.conditional_simulate): every curve of a
multi-series drawn at its own times given its data, npaths paths per curve, in one call.

  * a one-curve multi-series draws what Series(curve).simulate draws from the same random numbers;
  * a draw depends only on (seed, path, global curve index, theta row): not on batch mates, npaths, path chunking,
    or whether the theta row was given per curve or per path -- bit for bit;
  * the draws follow the exact Gaussian-process conditional law, and agree with MultiSeries.predict at scale;
  * rejected theta rows, curves without times, 2-point curves and draws at data times."""
import numpy as np
import pytest

from test_gpu_survey_filter import _explicit, _models, _ragged_survey, _thetas

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def C():
    import carma_pack_b200 as c
    if c._lib.device_count() < 1:
        pytest.fail("no CUDA device visible: GPU tests must run on the B200 box")
    return c


def _times(rng, t):
    """Backcasts, gaps, data times, duplicates and forecasts of one curve, unsorted."""
    span = t[-1] - t[0]
    q = [t[0] - rng.uniform(0.5, 2.0) * span, t[0] - 0.3, t[0], t[t.size // 2], t[t.size // 2], t[-1],
         t[-1] + 0.5, t[-1] + rng.uniform(0.5, 2.0) * span]
    q += list(rng.uniform(t[0], t[-1], 5))
    q.append(q[-1])
    q = np.array(q)
    return q[rng.permutation(q.size)]


def _queries(rng, ts, empty=()):
    qs = [np.zeros(0) if c in empty else _times(rng, t) for c, t in enumerate(ts)]
    return qs, np.cumsum([0] + [x.size for x in qs])


def _one_curve(C, ts, ys, es, c):
    return C.MultiSeries(ts[c], ys[c], es[c], [0, ts[c].size])


@pytest.mark.parametrize("model", range(7))
def test_one_curve_survey_matches_the_single_series_draw(C, model):
    """Same Philox counters as carma_simulate, same merge of data and requested times: the two differ only by the
    forward filter (time-parallel scan against the sequential recursion) and by the theta transform against the
    explicit parameters.  Both are rounding, amplified at most by the conditioning of the curve: 1e-6 relative to the
    curve's scale, where a different random number would move a draw by O(1)."""
    m, ts, ys, es = _ragged_survey(C, seed=21)
    name, kind, p, q, tail = _models(C)[model]
    th = _thetas(ys, tail, seed=40 + model, bad=False)
    pri = m.default_priors()
    rng = np.random.default_rng(model)
    qs, qo = _queries(rng, ts)
    ll = m.loglik(kind, p, q, th, flags=m._default_flags(p, None))
    npaths, seed = 3, 1234 + model
    checked = 0
    for c in range(m.ncurves):
        if not np.isfinite(ll[c]):
            continue
        one = _one_curve(C, ts, ys, es, c)
        got = one.conditional_simulate(kind, p, q, th[c:c + 1], qs[c], [0, qs[c].size], npaths=npaths, seed=seed)
        one.close()
        t, y, e = m.curve(c)
        s2, roots, ma = _explicit(C, kind, p, q, th[c], C.Prior(*pri[c]))
        s = C.Series(t, y, e)
        want = s.simulate(s2, roots, ma, qs[c] - ts[c][0], measerr_scale=th[c, 1], mu=th[c, 2], seed=seed,
                          npaths=npaths)
        s.close()
        assert got.shape == want.shape == (npaths, qs[c].size)
        scale = max(np.std(ys[c]), 1.0)
        np.testing.assert_allclose(got, want, rtol=0, atol=1e-6 * scale, err_msg="%s curve %d" % (name, c))
        checked += 1
    assert checked >= m.ncurves // 2, checked
    m.close()


def test_draws_do_not_depend_on_batch_mates_npaths_chunks_or_theta_layout(C, monkeypatch):
    m, ts, ys, es = _ragged_survey(C, seed=22)
    name, kind, p, q, tail = _models(C)[2]
    th = _thetas(ys, tail, seed=5, bad=False)
    rng = np.random.default_rng(3)
    qs, qo = _queries(rng, ts, empty=(7,))
    tq = np.concatenate(qs)
    seed = 77
    full = m.conditional_simulate(kind, p, q, th, tq, qo, npaths=7, seed=seed)
    assert full.shape == (7, tq.size) and np.all(np.isfinite(full))
    # curve c of the survey is the one-curve survey of that curve with curve_offset = c
    for c in (0, 4, 12, 18):
        one = _one_curve(C, ts, ys, es, c)
        np.testing.assert_array_equal(one.conditional_simulate(kind, p, q, th[c:c + 1], qs[c], [0, qs[c].size],
                                                               npaths=7, seed=seed, curve_offset=c),
                                      full[:, qo[c]:qo[c + 1]])
        one.close()
    # path j does not depend on npaths
    many = m.conditional_simulate(kind, p, q, th, tq, qo, npaths=500, seed=seed)
    np.testing.assert_array_equal(many[:7], full)
    # several path chunks give the bits of one chunk
    monkeypatch.setenv("CARMA_MULTI_SIMULATE_BUDGET", "1")      # one path per chunk
    np.testing.assert_array_equal(m.conditional_simulate(kind, p, q, th, tq, qo, npaths=7, seed=seed), full)
    monkeypatch.setenv("CARMA_MULTI_SIMULATE_BUDGET", str(40 * 8 * (m.offsets[-1] + 13 * tq.size)))   # < 40 per chunk
    np.testing.assert_array_equal(m.conditional_simulate(kind, p, q, th, tq, qo, npaths=500, seed=seed), many)
    monkeypatch.delenv("CARMA_MULTI_SIMULATE_BUDGET")
    # per-path theta equal to the per-curve row: the per-curve call
    per_path = np.repeat(th[:, None, :], 7, axis=1)
    np.testing.assert_array_equal(m.conditional_simulate(kind, p, q, per_path, tq, qo, npaths=7, seed=seed), full)
    # path j of a per-path call is path j of a per-curve call with theta[:, j, :]
    per_path = np.stack([_thetas(ys, tail, seed=100 + j, bad=False) for j in range(4)], axis=1)
    got = m.conditional_simulate(kind, p, q, per_path, tq, qo, npaths=4, seed=seed)
    for j in range(4):
        np.testing.assert_array_equal(got[j], m.conditional_simulate(kind, p, q, per_path[:, j, :], tq, qo, npaths=j + 1,
                                                                     seed=seed)[j])
    # a different seed or curve_offset gives different draws
    assert not np.any(m.conditional_simulate(kind, p, q, th, tq, qo, npaths=7, seed=seed + 1) == full)
    assert not np.any(m.conditional_simulate(kind, p, q, th, tq, qo, npaths=7, seed=seed, curve_offset=1) == full)
    m.close()


def _kernel(C, sigsqr, roots, ma):
    from carma_pack_b200 import synth
    return lambda a, b: np.array([[synth.carma_variance(sigsqr, roots, ma, lag=abs(x - z)) for z in b] for x in a])


@pytest.mark.parametrize("model", [0, 2, 3, 4])
def test_draws_follow_the_exact_gaussian_process_conditional(C, model):
    """4,000 paths per curve of a small ragged survey, whitened with the dense conditional mean and covariance of the
    Gaussian process (carma_variance as the kernel): white N(0, 1) within Monte-Carlo error."""
    lengths = [2, 5, 38, 3, 80, 21, 9, 60]
    m, ts, ys, es = _ragged_survey(C, seed=30 + model, lengths=lengths)
    name, kind, p, q, tail = _models(C)[model]
    th = _thetas(ys, tail, seed=50 + model, bad=False)
    pri = m.default_priors()
    rng = np.random.default_rng(10 + model)
    qs, qo = _queries(rng, ts)
    n = 4000
    sims = m.conditional_simulate(kind, p, q, th, np.concatenate(qs), qo, npaths=n, seed=9)
    assert sims.shape == (n, qo[-1])
    ll = m.loglik(kind, p, q, th, flags=m._default_flags(p, None))
    assert np.isfinite(ll).sum() >= 4, ll
    for c in range(m.ncurves):
        if not np.isfinite(ll[c]):                   # outside the curve's prior (short curves, CAR(1))
            continue
        assert np.all(np.isfinite(sims[:, qo[c]:qo[c + 1]])), (name, c)
        s2, roots, ma = _explicit(C, kind, p, q, th[c], C.Prior(*pri[c]))
        mu, scale = th[c, 2], th[c, 1]
        kern = _kernel(C, s2, roots, ma)
        t, tsim = ts[c], qs[c]
        Kdd = kern(t, t) + np.diag(scale * es[c] ** 2)
        Ksd = kern(tsim, t)
        cmean = mu + Ksd @ np.linalg.solve(Kdd, ys[c] - mu)
        ccov = kern(tsim, tsim) - Ksd @ np.linalg.solve(Kdd, Ksd.T)
        x = sims[:, qo[c]:qo[c + 1]]
        at_data = np.isin(tsim, t)
        assert np.all(x[:, at_data].std(axis=0) > 0), (name, c)     # the draw at a data time is not the datum
        w, V = np.linalg.eigh(ccov)
        keep = w > 1e-9 * w.max()
        white = (x - cmean) @ V[:, keep] / np.sqrt(w[keep])
        assert np.all(np.abs(white.mean(axis=0)) < 4.5 / np.sqrt(n)), (name, c, np.abs(white.mean(axis=0)).max())
        cov = np.cov(white.T)
        assert np.all(np.abs(np.diag(cov) - 1.0) < 5.0 * np.sqrt(2.0 / n)), (name, c, np.abs(np.diag(cov) - 1.0).max())
        off = cov - np.diag(np.diag(cov))
        assert np.abs(off).max() < 5.5 / np.sqrt(n), (name, c, np.abs(off).max())
    m.close()


def test_sample_moments_agree_with_predict_at_scale(C):
    """300 simulated curves x 2,000 paths: per query, the sample mean is predict's qmean + mu within 5.5 standard errors
    (sqrt(qvar / n)) and the sample variance is qvar within 5.5 standard errors (qvar sqrt(2 / (n - 1)))."""
    from carma_pack_b200 import synth
    nc, ny, n = 300, 400, 2000
    th0 = synth.carma31_theta(sigmay=1.5, mu=2.0)
    m = C.MultiSeries.simulate(nc, ny, C.KIND_CARMA, 3, 1, th0, yerr=0.2, dt_min=0.05, dt_max=20.0, seed=4)
    span = m.curve_stats()["tspan"]
    rng = np.random.default_rng(6)
    nq = 12
    tq = (rng.uniform(-0.1, 1.1, (nc, nq)) * span[:, None]).reshape(-1)
    qo = np.arange(nc + 1, dtype=np.int64) * nq
    th = np.tile(th0, (nc, 1))
    qm, qv = m.predict(C.KIND_CARMA, 3, 1, th, tq, qo)
    sims = m.conditional_simulate(C.KIND_CARMA, 3, 1, th, tq, qo, npaths=n, seed=2)
    assert sims.shape == (n, tq.size) and np.all(np.isfinite(sims))
    zm = (sims.mean(axis=0) - qm) / np.sqrt(qv / n)
    zv = (sims.var(axis=0, ddof=1) - qv) / (qv * np.sqrt(2.0 / (n - 1)))
    assert np.abs(zm).max() < 5.5, np.abs(zm).max()
    assert np.abs(zv).max() < 5.5, np.abs(zv).max()
    assert 0.85 < zm.std() < 1.15 and 0.85 < zv.std() < 1.15, (zm.std(), zv.std())
    m.close()


def test_rejected_rows_empty_curves_and_short_curves(C):
    m, ts, ys, es = _ragged_survey(C, seed=23)
    assert min(t.size for t in ts) == 2
    name, kind, p, q, tail = _models(C)[3]
    th = _thetas(ys, tail, seed=8, bad=False)
    rng = np.random.default_rng(4)
    qs, qo = _queries(rng, ts, empty=(2, 9))
    tq = np.concatenate(qs)
    # sigma_y < 0 fails the prior bounds (flags = 0): curve 4 is rejected by the transform, and only curve 4
    good = m.conditional_simulate(kind, p, q, th, tq, qo, npaths=5, seed=3, flags=0)
    in4 = np.zeros(tq.size, bool)
    in4[qo[4]:qo[5]] = True
    assert np.all(np.isfinite(good[:, in4]))
    bad = th.copy()
    bad[4, 0] = -1.0
    got = m.conditional_simulate(kind, p, q, bad, tq, qo, npaths=5, seed=3, flags=0)
    assert np.all(np.isnan(got[:, in4]))
    np.testing.assert_array_equal(got[:, ~in4], good[:, ~in4])
    # per path: a rejected row NaNs exactly that path of that curve
    per_path = np.repeat(th[:, None, :], 5, axis=1)
    per_path[8, 2, 0] = -1.0
    got = m.conditional_simulate(kind, p, q, per_path, tq, qo, npaths=5, seed=3, flags=0)
    mask = np.zeros(got.shape, bool)
    mask[2, qo[8]:qo[9]] = True
    assert np.all(np.isfinite(good[mask])) and np.all(np.isnan(got[mask]))
    np.testing.assert_array_equal(got[~mask], good[~mask])
    # the default flags (IGNORE_BOUNDS for p > 1): every curve is drawn, including the 2-point ones
    assert np.all(np.isfinite(m.conditional_simulate(kind, p, q, th, tq, qo, npaths=5, seed=3)))
    # no times at all, and no paths: nothing to do
    none = m.conditional_simulate(kind, p, q, th, np.zeros(0), np.zeros(m.ncurves + 1, np.int64), npaths=3, seed=1)
    assert none.shape == (3, 0)
    m.close()


def test_argument_checks(C):
    m, ts, ys, es = _ragged_survey(C, seed=24, lengths=[5, 7, 9])
    name, kind, p, q, tail = _models(C)[2]
    th = _thetas(ys, tail, seed=1, bad=False)
    L = C._lib.lib
    tq = np.array([1.0, 2.0, 3.0, 4.0])
    out = np.zeros(64)

    def call(so, t=tq, rows=3, npaths=2, curve_offset=0, theta=th):
        so = np.asarray(so, np.int64)
        return L.carma_multi_simulate(m.handle, kind, p, q, None, theta.ctypes.data, rows, 0, so.ctypes.data, t.ctypes.data,
                                      npaths, 1, curve_offset, out.ctypes.data)

    assert call([0, 1, 2, 4]) == 0
    for args, word in ((([0, 3, 2, 4],), b"non-decreasing"), (([0, 1, 2, 4], np.array([1.0, np.nan, 3.0, 4.0])), b"non-finite"),
                       (([0, 1, 2, 4], np.array([1.0, np.inf, 3.0, 4.0])), b"non-finite")):
        assert call(*args) == 1
        assert b"carma_multi_simulate" in L.carma_last_error() and word in L.carma_last_error()
    for rows in (2, 4, 5):
        assert call([0, 1, 2, 4], rows=rows) == 1 and b"theta_rows" in L.carma_last_error()
    assert call([0, 1, 2, 4], rows=6, theta=np.repeat(th, 2, axis=0)) == 0
    assert call([0, 1, 2, 4], curve_offset=2 ** 32 - 3) == 0
    assert call([0, 1, 2, 4], curve_offset=2 ** 32 - 2) == 1 and b"2^32" in L.carma_last_error()
    assert call([0, 1, 2, 4], npaths=0) == 0
    with pytest.raises(ValueError):
        m.conditional_simulate(kind, p, q, th, tq, [0, 1, 4])
    with pytest.raises(ValueError):
        m.conditional_simulate(kind, p, q, th[:2], tq, [0, 1, 2, 4])
    with pytest.raises(ValueError):
        m.conditional_simulate(kind, p, q, np.repeat(th[:, None, :], 3, axis=1), tq, [0, 1, 2, 4], npaths=2)
    m.close()
