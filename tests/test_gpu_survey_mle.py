"""Survey-scale maximum likelihood (carma_multi_mle_grid_device, MultiSeries.get_mle / choose_order): every curve of a
multi-series fitted, for every model, in one launch.

  * every curve's fits equal those of a Series built from that curve alone, bit for bit (and through
    test_device_optimizer_matches_the_host_loop, the host loop's);
  * a curve's starts and fits do not depend on its batch mates or on how the survey is split (curve_offset);
  * the Python layer builds the starts and boxes CarmaModel builds for the same curve;
  * on a simulated survey the fits reach at least the likelihood of the true parameters;
  * the per-curve AICc table is the reference's formula applied to the per-model fits."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def C():
    import carma_pack_b200 as c
    if c._lib.device_count() < 1:
        pytest.fail("no CUDA device visible: GPU tests must run on the B200 box")
    return c


def _kind(C, p, q):
    return C.KIND_CAR1 if p == 1 else (C.KIND_CARMA if q > 0 else C.KIND_CARP)


def _ragged_survey(C, seed=8):
    """12 short curves whose first points sit at every offset mod 4 of the CSR arrays, plus one of 3,000 points (too
    long for a warp's shared-memory slice)."""
    from carma_pack_b200 import synth
    rng = np.random.default_rng(seed)
    ar, ma, s2 = synth.carma31_truth()
    lengths = [5, 38, 400, 121, 9, 250, 63, 302, 18, 3000, 199, 77, 6]
    ts, ys, es, off = [], [], [], [0]
    for ny in lengths:
        t = np.cumsum(rng.uniform(0.2, 3.0, ny)) + rng.uniform(0, 50)
        y = 2.0 + synth.carma_process(t, s2, ar, ma, rng) + 0.2 * rng.standard_normal(ny)
        ts.append(t); ys.append(y); es.append(rng.uniform(0.1, 0.3, ny)); off.append(off[-1] + ny)
    assert {o % 4 for o in off[:-1]} == {0, 1, 2, 3}
    m = C.MultiSeries(np.concatenate(ts), np.concatenate(ys), np.concatenate(es), off)
    return m, ts, ys, es


def test_every_curve_equals_its_own_series_bitwise(C):
    from carma_pack_b200.carma_pack import mle_bounds
    m, ts, ys, es = _ragged_survey(C)
    nc = m.ncurves
    st = m.curve_stats()
    assert list(st["ny"]) == [t.size for t in ts]
    for c in range(nc):
        dt = np.diff(ts[c])
        assert st["min_dt"][c] == dt.min() and st["dt_max"][c] == dt.max()
        assert st["tspan"][c] == ts[c][-1] - ts[c][0]
    pri = m.default_priors()
    pri["max_stdev"] *= 1.5          # priors given by the caller, not the defaults
    rng = np.random.default_rng(5)
    jobs = []
    for p, q, ns in ((1, 0, 12), (2, 0, 8), (3, 1, 16), (5, 2, 10), (3, 0, 0)):
        kind = _kind(C, p, q)
        lo, hi = mle_bounds(p, q, np.sqrt(st["y_var_pop"]), st["min_dt"], st["tspan"])
        d = lo.shape[1]
        x0 = np.empty((nc, ns, d))
        for c in range(nc):
            fin = np.isfinite(lo[c])
            x0[c][:, fin] = rng.uniform(lo[c][fin], hi[c][fin], (ns, fin.sum()))
            x0[c][:, ~fin] = rng.normal(0.0, 1.0, (ns, (~fin).sum()))
            x0[c][:, 2] += st["y_mean"][c]
        jobs.append((kind, p, q, x0, lo, hi, 0 if p == 1 else C.IGNORE_BOUNDS))
    grid = m.mle_grid(jobs, priors=pri, maxiter=300)
    assert len(grid) == len(jobs)
    for (kind, p, q, x0, lo, hi, flags), (x, f, nit, nfev) in zip(jobs, grid):
        assert x.shape == x0.shape and f.shape == x0.shape[:2] and nit.shape == nfev.shape == (nc,)
        if x0.shape[1] == 0:
            assert np.all(nit == 0) and np.all(nfev == 0)
            continue
        for c in range(nc):
            s = C.Series(ts[c], ys[c], es[c])
            x1, f1, nit1, nfev1 = s.mle_batch(kind, p, q, x0[c], lo[c], hi[c], prior=C.Prior(*pri[c]), flags=flags,
                                              maxiter=300, on_device=True)
            np.testing.assert_array_equal(x[c], x1)
            np.testing.assert_array_equal(f[c], f1)
            assert (nit[c], nfev[c]) == (nit1, nfev1), (p, q, c)
            s.close()
        assert np.sum(f < 1e299) >= 0.75 * f.size
    assert m.mle_grid([]) == []
    m.close()


def test_fits_do_not_depend_on_batch_mates_or_sharding(C):
    m, ts, ys, es = _ragged_survey(C, seed=9)
    full = m.get_mle(3, 1, ntrials=8, seed=123, maxiter=300)
    k, n = 4, 5
    off = np.cumsum([0] + [t.size for t in ts[k:k + n]])
    part = C.MultiSeries(np.concatenate(ts[k:k + n]), np.concatenate(ys[k:k + n]), np.concatenate(es[k:k + n]), off)
    sub = part.get_mle(3, 1, ntrials=8, seed=123, maxiter=300, curve_offset=k)
    for key in ("x0", "lower", "upper", "all_x", "all_fun", "x", "fun", "nit", "nfev"):
        np.testing.assert_array_equal(np.asarray(sub[key]), np.asarray(full[key])[k:k + n], err_msg=key)
    part.close()
    m.close()


def test_python_layer_matches_the_single_curve_api(C):
    m, ts, ys, es = _ragged_survey(C, seed=10)
    keep = [c for c in range(m.ncurves) if ts[c].size >= 30]
    m.close()
    ts, ys, es = [ts[c] for c in keep], [ys[c] for c in keep], [es[c] for c in keep]
    m = C.MultiSeries(np.concatenate(ts), np.concatenate(ys), np.concatenate(es), np.cumsum([0] + [t.size for t in ts]))
    ntrials, seed = 6, 77
    for p, q in ((1, 0), (3, 1)):
        res = m.get_mle(p, q, ntrials=ntrials, seed=seed, maxiter=200)
        for c in range(m.ncurves):
            model = C.CarmaModel(ts[c], ys[c], es[c])
            kind, x0, lo, hi, prior, flags = model.mle_starts(p, q, ntrials, seed, trial_offset=c * ntrials)
            np.testing.assert_allclose(res.x0[c], x0, rtol=1e-12)
            np.testing.assert_allclose(res.lower[c], lo, rtol=1e-12)
            np.testing.assert_allclose(res.upper[c], hi, rtol=1e-12)
        np.testing.assert_array_equal(res.fun, res.all_fun.min(axis=1))
        best = np.argmin(res.all_fun, axis=1)
        np.testing.assert_array_equal(res.x, res.all_x[np.arange(m.ncurves), best])
        assert np.all(res.success) and np.all(res.nit >= 1) and np.all(res.nfev > 0)
    m.close()


def test_fits_reach_the_likelihood_of_the_truth_on_a_simulated_survey(C):
    from carma_pack_b200 import synth
    th = synth.carma31_theta()
    nc = 64
    m = C.MultiSeries.simulate(nc, 300, C.KIND_CARMA, 3, 1, th, yerr=0.2, dt_min=0.05, dt_max=60.0, seed=21)
    res = m.get_mle(3, 1, ntrials=16, seed=4)
    inside = np.all((th >= res.lower) & (th <= res.upper), axis=1)
    assert inside.all()
    f_true = -m.loglik(C.KIND_CARMA, 3, 1, np.tile(th, (nc, 1)), priors=m.default_priors(), flags=C.IGNORE_BOUNDS)
    assert np.all(np.isfinite(f_true))
    ok = res.fun <= f_true + 1e-6 * np.abs(res.fun)
    assert ok.mean() >= 0.95, (ok.mean(), (res.fun - f_true)[~ok])
    m.close()


def test_choose_order_table_is_the_formula_on_the_per_model_fits(C):
    from carma_pack_b200.carma_pack import aicc
    from carma_pack_b200 import synth
    m = C.MultiSeries.simulate(8, 120, C.KIND_CARMA, 3, 1, synth.carma31_theta(), yerr=0.2, dt_min=0.05, dt_max=60.0,
                               seed=3)
    best_pq, pqlist, table, mles = m.choose_order(3, ntrials=8, seed=1000)
    assert pqlist == [(1, 0), (2, 0), (2, 1), (3, 0), (3, 1), (3, 2)]
    assert table.shape == (8, len(pqlist)) and best_pq.shape == (8, 2)
    ny = m.curve_stats()["ny"]
    for k, (p, q) in enumerate(pqlist):
        alone = m.get_mle(p, q, ntrials=8, seed=1000 + k)
        np.testing.assert_array_equal(alone.all_fun, mles[k].all_fun)
        np.testing.assert_array_equal(table[:, k], aicc(alone.fun, p, q, ny))
        np.testing.assert_array_equal(table[:, k], 2.0 * (2 + p + q) + 2.0 * alone.fun +
                                      2.0 * (2 + p + q) * (3.0 + p + q) / (ny - (2 + p + q) - 1.0))
    np.testing.assert_array_equal(best_pq, np.asarray(pqlist)[np.argmin(table, axis=1)])
    m.close()
