"""Survey-scale Kalman filter, fit diagnostics and prediction (carma_multi_filter / _assess_fit / _predict,
MultiSeries.kalman_filter / assess_fit_values / predict): every curve of a multi-series in one launch.

  * the per-curve log-density is bitwise MultiSeries.loglik's (-inf and NaN rows included);
  * mean / var of every curve agree with a Series built from that curve, and with the oracle;
  * a curve's outputs do not depend on its batch mates;
  * the residual moments and ACFs are numpy's on the downloaded residuals, and white at the true parameters;
  * predictions agree with Series.predict and the oracle for backcasts, forecasts, data times, duplicates and unsorted
    times, come back in caller order, and do not depend on where the curves' time axes start;
  * the filter scores fitted parameters exactly as the survey fits did."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def C():
    import carma_pack_b200 as c
    if c._lib.device_count() < 1:
        pytest.fail("no CUDA device visible: GPU tests must run on the B200 box")
    return c


@pytest.fixture(scope="module")
def O():
    from oracle import oracle
    oracle.build()
    return oracle


LENGTHS = [2, 5, 38, 3, 400, 121, 9, 4, 250, 63, 302, 18, 3000, 199, 77, 6, 7, 8, 11]


def _ragged_survey(C, seed=8, lengths=LENGTHS):
    """Curves of 2 to 3,000 points whose first points sit at every offset mod 4 of the CSR arrays (every head peel and
    tail of the block stores), absolute times starting anywhere in [0, 50)."""
    from carma_pack_b200 import synth
    rng = np.random.default_rng(seed)
    ar, ma, s2 = synth.carma31_truth()
    ts, ys, es, off = [], [], [], [0]
    for ny in lengths:
        t = np.cumsum(rng.uniform(0.2, 3.0, ny)) + rng.uniform(0, 50)
        y = 2.0 + synth.carma_process(t, s2, ar, ma, rng) + 0.2 * rng.standard_normal(ny)
        ts.append(t); ys.append(y); es.append(rng.uniform(0.1, 0.3, ny)); off.append(off[-1] + ny)
    assert lengths is not LENGTHS or {o % 4 for o in off[:-1]} == {0, 1, 2, 3}
    m = C.MultiSeries(np.concatenate(ts), np.concatenate(ys), np.concatenate(es), off)
    return m, ts, ys, es


def _logquad(roots):
    from carma_pack_b200 import synth
    return list(synth.roots_to_logquad(roots))


# (name, kind, p, q, theta tail after (sigma_y, scale, mu))
def _models(C):
    return [
        ("car1", C.KIND_CAR1, 1, 0, [np.log(0.3)]),
        ("car2", C.KIND_CARP, 2, 0, _logquad([-0.1 + 0.5j, -0.1 - 0.5j])),
        ("carma31_conj", C.KIND_CARMA, 3, 1, _logquad([-0.05 + 0.3j, -0.05 - 0.3j, -0.4]) + [np.log(2.0)]),
        ("carma31_real", C.KIND_CARMA, 3, 1, _logquad([-0.1, -0.7, -0.3]) + [np.log(2.0)]),
        ("carma53", C.KIND_CARMA, 5, 3, _logquad([-0.05 + 0.3j, -0.05 - 0.3j, -0.2, -0.9, -0.4]) +
         _logquad([-1.5 + 0.5j, -1.5 - 0.5j, -3.0])),
        ("carma76", C.KIND_CARMA, 7, 6, _logquad([-0.05 + 0.3j, -0.05 - 0.3j, -0.1 + 1.1j, -0.1 - 1.1j, -0.3, -0.8, -0.5]) +
         _logquad([-1.5 + 0.5j, -1.5 - 0.5j, -2.0, -4.0, -3.0 + 1.0j, -3.0 - 1.0j])),
        ("zcarma5", C.KIND_ZCARMA, 5, 0, _logquad([-0.05 + 0.3j, -0.05 - 0.3j, -0.2, -0.9, -0.4]) + [0.3]),
    ]


def _thetas(ys, tail, seed, bad=True):
    """One theta row per curve around the model, scaled to the curve; with bad=True one row outside the prior (negative
    sigma_y) and one NaN row."""
    rng = np.random.default_rng(seed)
    rows = []
    for y in ys:
        head = [np.std(y) * rng.uniform(0.8, 1.2), rng.uniform(1.0, 1.2), np.mean(y)]
        rows.append(head + list(np.asarray(tail) + rng.normal(0.0, 0.02, len(tail))))
    th = np.array(rows)
    if bad:
        th[1, 0] = -1.0
        th[4, 3] = np.nan
    return th


def _explicit(C, kind, p, q, th, prior):
    der = C._lib.derived_params(kind, p, q, th[None, :], prior=prior)
    return der["sigma"][0] ** 2, der["ar_roots"][0], der["ma_coefs"][0]


@pytest.mark.parametrize("model", range(7))
def test_filter_matches_k4_single_curve_and_oracle(C, O, model):
    m, ts, ys, es = _ragged_survey(C)
    name, kind, p, q, tail = _models(C)[model]
    th = _thetas(ys, tail, seed=model)
    pri = m.default_priors()
    for flags in ((0, C.IGNORE_BOUNDS) if p > 1 else (0,)):
        mean, var, ll = m.kalman_filter(kind, p, q, th, flags=flags)
        want = m.loglik(kind, p, q, th, priors=pri, flags=flags)
        np.testing.assert_array_equal(ll, want, err_msg=name)            # bitwise, -inf and NaN rows included
        if flags == 0:
            assert ll[1] == -np.inf                   # sigma_y < 0 fails the prior bounds
    assert not np.isfinite(ll[4])
    ll_default = m.kalman_filter(kind, p, q, th)[2]
    np.testing.assert_array_equal(ll_default, m.loglik(kind, p, q, th, flags=0 if p == 1 else C.IGNORE_BOUNDS))
    off = m.offsets
    for c in range(m.ncurves):
        mc, vc = mean[off[c]:off[c + 1]], var[off[c]:off[c + 1]]
        if ll[c] == -np.inf:                          # rejected by the transform: the whole curve is NaN
            assert np.all(np.isnan(mc)) and np.all(np.isnan(vc)), (name, c)
            continue
        if np.isnan(ll[c]):                           # accepted, NaN through the recursion
            assert np.isnan(vc[-1]), (name, c)
            continue
        t, y, e = m.curve(c)
        s2, roots, ma = _explicit(C, kind, p, q, th[c], C.Prior(*pri[c]))
        s = C.Series(t, y, e)
        sm, sv = s.filter(s2, roots, ma, measerr_scale=th[c, 1], mu=th[c, 2])
        s.close()
        assert mc[0] - th[c, 2] == 0.0
        np.testing.assert_allclose(mc - th[c, 2], sm, rtol=0, atol=1e-9, err_msg="%s curve %d" % (name, c))
        np.testing.assert_allclose(vc, sv, rtol=1e-9, err_msg="%s curve %d" % (name, c))
        if c in (0, 5, 12):
            om, ov = O.filterp(t, y - th[c, 2], np.sqrt(th[c, 1]) * e, s2, roots, ma)
            np.testing.assert_allclose(mc - th[c, 2], om, rtol=0, atol=1e-9)
            np.testing.assert_allclose(vc, ov, rtol=1e-9)
    m.close()


def test_block_and_scalar_stores_agree_bitwise(C, monkeypatch):
    m, ts, ys, es = _ragged_survey(C, seed=3)
    name, kind, p, q, tail = _models(C)[2]
    th = _thetas(ys, tail, seed=11)
    a = m.kalman_filter(kind, p, q, th)
    monkeypatch.setenv("CARMA_MULTI_FILTER_STORES", "scalar")
    b = m.kalman_filter(kind, p, q, th)
    for x, y in zip(a, b):
        np.testing.assert_array_equal(x, y)
    m.close()


def test_outputs_do_not_depend_on_batch_mates(C):
    m, ts, ys, es = _ragged_survey(C, seed=9)
    name, kind, p, q, tail = _models(C)[4]
    th = _thetas(ys, tail, seed=4, bad=False)
    mean, var, ll = m.kalman_filter(kind, p, q, th)
    k, n = 9, 6
    off = np.cumsum([0] + [t.size for t in ts[k:k + n]])
    part = C.MultiSeries(np.concatenate(ts[k:k + n]), np.concatenate(ys[k:k + n]), np.concatenate(es[k:k + n]), off)
    pm, pv, pll = part.kalman_filter(kind, p, q, th[k:k + n])
    lo, hi = m.offsets[k], m.offsets[k + n]
    np.testing.assert_array_equal(pm, mean[lo:hi])
    np.testing.assert_array_equal(pv, var[lo:hi])
    np.testing.assert_array_equal(pll, ll[k:k + n])
    fa, fp = m.assess_fit_values(kind, p, q, th, nlags=1), part.assess_fit_values(kind, p, q, th[k:k + n], nlags=1)
    for key in ("loglik", "resid_mean", "resid_std", "acf", "acf_sq"):
        np.testing.assert_array_equal(fp[key], fa[key][k:k + n], err_msg=key)
    part.close()
    m.close()


def _acf(x, nlags):
    x = x - x.mean()
    full = np.correlate(x, x, mode="full")[x.size - 1:]
    return full[1:nlags + 1] / full[0]


@pytest.mark.parametrize("nlags", [1, 20, 40, 100])
def test_assess_fit_equals_numpy_on_the_residuals(C, nlags):
    lengths = LENGTHS if nlags == 1 else [n for n in LENGTHS if n > 100] + [101, 102, 103, 104]
    m, ts, ys, es = _ragged_survey(C, seed=12, lengths=lengths)
    name, kind, p, q, tail = _models(C)[3]
    th = _thetas(ys, tail, seed=7, bad=False)
    mean, var, ll = m.kalman_filter(kind, p, q, th)
    res = m.assess_fit_values(kind, p, q, th, nlags=nlags)
    assert res.acf.shape == res.acf_sq.shape == (m.ncurves, nlags)
    np.testing.assert_array_equal(res.loglik, ll)
    off = m.offsets
    for c in range(m.ncurves):
        y = ys[c]
        r = (y - mean[off[c]:off[c + 1]]) / np.sqrt(var[off[c]:off[c + 1]])
        np.testing.assert_allclose(res.resid_mean[c], r.mean(), rtol=0, atol=1e-12)
        np.testing.assert_allclose(res.resid_std[c], r.std(), rtol=0, atol=1e-12)
        np.testing.assert_allclose(res.acf[c], _acf(r, nlags), rtol=0, atol=1e-12)
        np.testing.assert_allclose(res.acf_sq[c], _acf(r ** 2, nlags), rtol=0, atol=1e-12)
        assert res.bound[c] == 1.96 / np.sqrt(y.size)
    m.close()


def test_residuals_are_white_at_the_true_parameters(C):
    from carma_pack_b200 import synth
    th = synth.carma31_theta()
    nc, ny = 256, 500
    m = C.MultiSeries.simulate(nc, ny, C.KIND_CARMA, 3, 1, th, yerr=0.2, dt_min=0.05, dt_max=60.0, seed=31)
    res = m.assess_fit_values(C.KIND_CARMA, 3, 1, np.tile(th, (nc, 1)), nlags=20)
    assert np.all(np.isfinite(res.loglik))
    inside = np.abs(res.acf) < res.bound[:, None]
    assert 0.92 <= inside.mean() <= 0.98, inside.mean()
    assert abs(res.resid_std.mean() - 1.0) < 0.01 and np.all(np.abs(res.resid_std - 1.0) < 0.15)
    assert abs(res.resid_mean.mean()) < 0.02
    m.close()


def test_bad_nlags_are_rejected(C):
    m, ts, ys, es = _ragged_survey(C)
    name, kind, p, q, tail = _models(C)[2]
    th = _thetas(ys, tail, seed=1, bad=False)
    for nlags in (0, -3, 2, 5):   # the shortest curve has 2 points
        with pytest.raises(C.CarmaError, match="carma_multi_assess_fit"):
            m.assess_fit_values(kind, p, q, th, nlags=nlags)
    assert m.assess_fit_values(kind, p, q, th, nlags=1).acf.shape == (m.ncurves, 1)
    m.close()


def _queries(rng, t):
    """Backcasts, forecasts to 10x the span, data times, duplicates and interior times, shuffled."""
    span = t[-1] - t[0]
    q = [t[0] - rng.uniform(0, 2) * span, t[0] - 1e-6, t[0], t[-1], t[-1] + 1e-3, t[-1] + 10.0 * span,
         t[-1] + rng.uniform(0, 3) * span, t[t.size // 2], t[t.size // 2]]
    q += list(rng.uniform(t[0], t[-1], 6))
    q.append(q[-1])
    q = np.array(q)
    return q[rng.permutation(q.size)]


@pytest.mark.parametrize("model", [0, 1, 2, 3, 4, 6])
def test_predict_matches_single_curve_and_oracle(C, O, model):
    m, ts, ys, es = _ragged_survey(C, seed=14)
    name, kind, p, q, tail = _models(C)[model]
    th = _thetas(ys, tail, seed=20 + model, bad=False)
    th[1, 0] = -1.0                                   # a rejected row: NaN predictions
    pri = m.default_priors()
    rng = np.random.default_rng(model)
    qs = [_queries(rng, t) for t in ts]
    qs[7] = np.zeros(0)                               # a curve without queries
    qo = np.cumsum([0] + [x.size for x in qs])
    qm, qv = m.predict(kind, p, q, th, np.concatenate(qs), qo)
    ll = m.loglik(kind, p, q, th, flags=0 if p == 1 else C.IGNORE_BOUNDS)
    for c in range(m.ncurves):
        gm, gv = qm[qo[c]:qo[c + 1]], qv[qo[c]:qo[c + 1]]
        if not np.isfinite(ll[c]):
            assert np.all(np.isnan(gm)) and np.all(np.isnan(gv))
            continue
        if qs[c].size == 0:
            continue
        t, y, e = m.curve(c)
        tq = qs[c] - ts[c][0]
        s2, roots, ma = _explicit(C, kind, p, q, th[c], C.Prior(*pri[c]))
        s = C.Series(t, y, e)
        sm, sv = s.predict(s2, roots, ma, tq, measerr_scale=th[c, 1], mu=th[c, 2])
        s.close()
        np.testing.assert_allclose(gm - th[c, 2], sm, rtol=1e-7, atol=1e-9, err_msg="%s curve %d" % (name, c))
        np.testing.assert_allclose(gv, sv, rtol=1e-8, err_msg="%s curve %d" % (name, c))
        if c in (0, 5, 12):
            om, ov = O.predictp(t, y - th[c, 2], np.sqrt(th[c, 1]) * e, s2, roots, ma, tq)
            np.testing.assert_allclose(gm - th[c, 2], om, rtol=1e-7, atol=1e-9)
            np.testing.assert_allclose(gv, ov, rtol=1e-8)
    m.close()


def test_predict_at_data_times_and_shifted_axes(C):
    m, ts, ys, es = _ragged_survey(C, seed=15)
    name, kind, p, q, tail = _models(C)[2]
    th = _thetas(ys, tail, seed=2, bad=False)
    rng = np.random.default_rng(2)
    qs = [_queries(rng, t) for t in ts]
    qo = np.cumsum([0] + [x.size for x in qs])
    tq = np.concatenate(qs)
    qm, qv = m.predict(kind, p, q, th, tq, qo)
    # the same curves on axes starting at 0, queries shifted alike
    t0 = np.repeat([t[0] for t in ts], np.diff(qo))
    m0 = C.MultiSeries(np.concatenate([t - t[0] for t in ts]), np.concatenate(ys), np.concatenate(es), m.offsets)
    zm, zv = m0.predict(kind, p, q, th, tq - t0, qo)
    np.testing.assert_allclose(zm, qm, rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(zv, qv, rtol=1e-9)
    # queries exactly at the data times of a survey whose axes start at 0: Series.predict at the same times
    tq0 = np.concatenate([m0.curve(c)[0] for c in range(m0.ncurves)])
    qo0 = m0.offsets
    dm, dv = m0.predict(kind, p, q, th, tq0, qo0)
    for c in (0, 4, 12):
        t, y, e = m0.curve(c)
        s2, roots, ma = _explicit(C, kind, p, q, th[c], None)
        s = C.Series(t, y, e)
        sm, sv = s.predict(s2, roots, ma, t, measerr_scale=th[c, 1], mu=th[c, 2])
        s.close()
        np.testing.assert_allclose(dm[qo0[c]:qo0[c + 1]] - th[c, 2], sm, rtol=1e-7, atol=1e-9)
        np.testing.assert_allclose(dv[qo0[c]:qo0[c + 1]], sv, rtol=1e-8)
    # caller order: a permutation of the queries permutes the answers
    perm = rng.permutation(tq.size)
    curve_of = np.repeat(np.arange(m.ncurves), np.diff(qo))
    order = np.lexsort((perm, curve_of))              # permute within each curve
    pm_, pv_ = m.predict(kind, p, q, th, tq[order], qo)
    np.testing.assert_array_equal(pm_, qm[order])
    np.testing.assert_array_equal(pv_, qv[order])
    with pytest.raises(ValueError):
        m.predict(kind, p, q, th, tq, qo[:-1])
    m0.close()
    m.close()


def test_filter_scores_the_survey_fits(C):
    from carma_pack_b200 import synth
    nc = 32
    m = C.MultiSeries.simulate(nc, 300, C.KIND_CARMA, 3, 1, synth.carma31_theta(), yerr=0.2, dt_min=0.05, dt_max=60.0,
                               seed=5)
    fits = m.get_mle(3, 1, ntrials=8, seed=17)
    mean, var, ll = m.kalman_filter(C.KIND_CARMA, 3, 1, fits.x)
    np.testing.assert_allclose(ll, -fits.fun, rtol=1e-10)
    assert mean.shape == var.shape == (nc * 300,) and np.all(var > 0)
    m.close()
