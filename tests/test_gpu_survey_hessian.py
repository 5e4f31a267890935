"""Survey-scale fit uncertainties (carma_multi_hessian, MultiSeries.hessian, CarmaModel.hessian): gradient, Hessian and
Laplace covariance of every curve's log-density at its theta row, in one call.

  * loglik is bitwise MultiSeries.loglik (-inf and NaN rows included); rejected rows have status REJECTED and NaN
    elsewhere;
  * grad / hessian are the documented stencil evaluated with MultiSeries.loglik and assembled in numpy, and agree with
    the same stencil from the long-double CPU oracle within the loglik parity gap amplified by 1 / (h_i h_j);
  * H_mu,mu is -1^T K^-1 1 of the dense Gaussian process (the log-density is quadratic in mu);
  * H at rel_step and rel_step / 2 agree to O(h^2); cov is (-H)^-1 and stderr sqrt(diag(cov));
  * outputs are bitwise the same across curve subsets, batch mates, chunking, and CarmaModel(curve).hessian;
  * each status has its documented cause;
  * at the fits of thousands of simulated curves, (theta_hat - theta_true) / stderr is standard normal and the
    gradient is negligible on the scale of stderr.

Ceilings were set from a run on a B200 (DESIGN.md "Survey fit uncertainties"): the device assembly was bitwise numpy's
on the same stencil values; the loglik parity gap to the oracle at most 1.2e-13 x max|f|; H_mu,mu within 8.1e-12 of
the dense answer; cov (-H) - I within 1.9e-17 x cond(H); at the fits, z means -0.11 .. 0.09 (the sigma_y MLE's
finite-sample bias is the -0.11), z standard deviations 0.99 .. 1.03, |g_i| stderr_i at most 5.4e-5."""
import numpy as np
import pytest

from test_gpu_survey_filter import LENGTHS, _explicit, _models, _ragged_survey, _thetas  # noqa: F401
from test_survey_hessian_host import assemble, stencil_rows

pytestmark = pytest.mark.gpu

EPS = np.finfo(float).eps
ASSEMBLY_TOL = 1e-12   # x max|H| of the curve: numpy's assembly against the device's, on the same stencil values
PARITY_GAP = 2e-12     # x max|f|: the loglik parity gap to the long-double oracle the comparison allows
GRAD_AT_FIT = 1e-3     # |g_i| stderr_i at a fit: the gradient in units of the Laplace width


@pytest.fixture(scope="module")
def C():
    import carma_pack_b200 as c
    if c._lib.device_count() < 1:
        pytest.fail("no CUDA device visible: GPU tests must run on the B200 box")
    return c


def _flags(C, p):
    return 0 if p == 1 else C.IGNORE_BOUNDS


def _stencil_values(m, kind, p, q, th, flags, rel_step=2.0 ** -13):
    """f (nc, npts) of the documented stencil by d^2 + d + 1 calls of MultiSeries.loglik, and the steps (nc, d)."""
    rows, steps = zip(*[stencil_rows(t, rel_step) for t in th])
    rows = np.array(rows)
    f = np.stack([m.loglik(kind, p, q, np.ascontiguousarray(rows[:, k]), flags=flags) for k in range(rows.shape[1])],
                 axis=1)
    return f, np.array(steps), rows


@pytest.mark.parametrize("model", range(7))
def test_loglik_stencil_and_assembly(C, model):
    m, ts, ys, es = _ragged_survey(C)
    name, kind, p, q, tail = _models(C)[model]
    th = _thetas(ys, tail, seed=model)
    flags = _flags(C, p)
    r = m.hessian(kind, p, q, th)
    d = th.shape[1]
    assert r.grad.shape == (m.ncurves, d) and r.hessian.shape == r.cov.shape == (m.ncurves, d, d)
    ll = m.loglik(kind, p, q, th, flags=flags)
    np.testing.assert_array_equal(r.loglik, ll, err_msg=name)           # bitwise, -inf and NaN rows included
    np.testing.assert_array_equal(m.hessian(kind, p, q, th, flags=0).loglik, m.loglik(kind, p, q, th, flags=0))
    assert not np.isfinite(r.loglik[4]) and r.status[4] in (C.HESS_REJECTED, C.HESS_NONFINITE)   # NaN row
    f, steps, _ = _stencil_values(m, kind, p, q, th, flags)
    np.testing.assert_array_equal(r.step, steps)
    for c in range(m.ncurves):
        what = "%s curve %d" % (name, c)
        if r.loglik[c] == -np.inf:
            assert r.status[c] == C.HESS_REJECTED, what
            for key in ("grad", "hessian", "cov", "stderr"):
                assert np.all(np.isnan(r[key][c])), (what, key)
            continue
        if not np.all(np.isfinite(f[c])):
            assert r.status[c] == C.HESS_NONFINITE, what
            assert np.all(np.isnan(r.grad[c])) and np.all(np.isnan(r.hessian[c])) and np.all(np.isnan(r.cov[c]))
            continue
        assert r.status[c] in (C.HESS_OK, C.HESS_NOT_NEGDEF), what
        g, H = assemble(f[c], steps[c])
        scale = np.abs(H).max()
        assert np.abs(r.hessian[c] - H).max() <= ASSEMBLY_TOL * scale, what
        assert np.abs(r.grad[c] - g).max() <= ASSEMBLY_TOL * scale * steps[c].max(), what
        np.testing.assert_array_equal(r.hessian[c], r.hessian[c].T)
        negdef = np.linalg.eigvalsh(-r.hessian[c]).min() > 0
        assert (r.status[c] == C.HESS_OK) == negdef, what
        if r.status[c] == C.HESS_OK:                 # covariance
            cond = np.linalg.cond(r.hessian[c])
            err = np.abs(r.cov[c] @ -r.hessian[c] - np.eye(d)).max()
            assert err <= 1e-13 * cond, (what, err, cond)
            np.testing.assert_array_equal(r.stderr[c], np.sqrt(np.diag(r.cov[c])))
        else:
            assert np.all(np.isnan(r.cov[c])) and np.all(np.isnan(r.stderr[c])), what
    m.close()


@pytest.mark.parametrize("model", [0, 1, 2, 4, 6])
def test_against_the_long_double_oracle(C, model):
    """The same stencil from oracle.logdensity(long_double=True): the device values differ from it by the loglik parity
    gap delta, which the assembly amplifies by at most 4 delta / (h_i h_j) (the coefficients of H_ij sum to 8 / 2 h_i h_j,
    those of H_ii to 4 / h_i^2)."""
    from oracle import oracle as O
    O.build()
    m, ts, ys, es = _ragged_survey(C)
    name, kind, p, q, tail = _models(C)[model]
    th = _thetas(ys, tail, seed=model, bad=False)
    flags = _flags(C, p)
    r = m.hessian(kind, p, q, th)
    pri = m.default_priors()
    checked = 0
    for c in range(m.ncurves):
        if len(ts[c]) > 400 or r.status[c] not in (C.HESS_OK, C.HESS_NOT_NEGDEF):
            continue
        rows, h = stencil_rows(th[c])
        f = O.logdensity(kind, p, q, ts[c], ys[c], es[c], rows, prior=C.Prior(*pri[c]), ignore_prior=bool(flags),
                         long_double=True)
        g, H = assemble(f, h)
        gap = PARITY_GAP * np.abs(f).max()
        bound = 4.0 * gap / np.outer(h, h) + ASSEMBLY_TOL * np.abs(H).max()
        err = np.abs(r.hessian[c] - H)
        assert np.all(err <= bound), ("%s curve %d" % (name, c), (err / bound).max())
        assert np.all(np.abs(r.grad[c] - g) <= gap / h + ASSEMBLY_TOL * np.abs(g).max()), (name, c)
        checked += 1
    assert checked >= 10, checked
    m.close()


def _dense_K(C, kind, p, q, th, t, e, prior):
    from carma_pack_b200 import synth
    s2, roots, ma = _explicit(C, kind, p, q, th, prior)
    return synth.carma_variance(s2, roots, ma, lag=np.abs(t[:, None] - t[None, :])) + np.diag(th[1] * e ** 2)


@pytest.mark.parametrize("model", [0, 2, 4])
def test_mu_curvature_is_the_dense_gp_answer(C, model):
    """log p is exactly quadratic in mu, so the second difference has no truncation error: H_mu,mu = -1^T K^-1 1.  A
    large step (rel_step 2^-4, a sixteenth of sigma_y) keeps the roundoff amplification eps |f| / h_mu^2 near 1e-12."""
    m, ts, ys, es = _ragged_survey(C)
    name, kind, p, q, tail = _models(C)[model]
    th = _thetas(ys, tail, seed=model, bad=False)
    r = m.hessian(kind, p, q, th, rel_step=2.0 ** -4)
    pri = m.default_priors()
    checked = 0
    for c in range(m.ncurves):
        if len(ts[c]) > 400 or not np.isfinite(r.hessian[c, 2, 2]):
            continue
        t, y, e = ts[c], ys[c], es[c]
        K = _dense_K(C, kind, p, q, th[c], t, e, C.Prior(*pri[c]))
        one = np.ones(t.size)
        want = -one @ np.linalg.solve(K, one)
        assert abs(r.hessian[c, 2, 2] - want) <= 1e-9 * abs(want), (name, c, r.hessian[c, 2, 2], want)
        checked += 1
    assert checked >= 10, checked
    m.close()


@pytest.mark.parametrize("model", [0, 2, 4])
def test_richardson_halving_the_step(C, model):
    m, ts, ys, es = _ragged_survey(C)
    name, kind, p, q, tail = _models(C)[model]
    th = _thetas(ys, tail, seed=model, bad=False)
    a = m.hessian(kind, p, q, th)
    b = m.hessian(kind, p, q, th, rel_step=2.0 ** -14)
    np.testing.assert_array_equal(b.step, a.step / 2)
    for c in range(m.ncurves):
        if not (np.all(np.isfinite(a.hessian[c])) and np.all(np.isfinite(b.hessian[c]))):
            continue
        scale = np.abs(a.hessian[c]).max()
        # truncation O(h^2) ~ 1e-8 relative; roundoff eps |f| / h^2 grows fourfold at h / 2
        ceil = 1e-6 * scale + 64 * EPS * abs(a.loglik[c]) / np.outer(b.step[c], b.step[c])
        assert np.all(np.abs(a.hessian[c] - b.hessian[c]) <= ceil), (name, c)
    m.close()


def test_outputs_are_bitwise_invariant(C, monkeypatch):
    import carma_pack_b200 as cp
    m, ts, ys, es = _ragged_survey(C, seed=9)
    keys = ("loglik", "grad", "hessian", "cov", "stderr", "status", "step")
    for model in (0, 1, 2):
        name, kind, p, q, tail = _models(C)[model]
        th = _thetas(ys, tail, seed=model, bad=False)
        full = m.hessian(kind, p, q, th)
        # batch mates: every other curve's row changes
        th2 = th.copy()
        th2[1::2, 3:] += 0.05
        mates = m.hessian(kind, p, q, th2)
        for key in keys:
            np.testing.assert_array_equal(mates[key][0::2], full[key][0::2], err_msg=key)
        # several chunks: three curves per chunk
        d = th.shape[1]
        monkeypatch.setenv("CARMA_MULTI_HESSIAN_BUDGET", str(3 * 8 * (d * d + d + 1)))
        ch = m.hessian(kind, p, q, th)
        monkeypatch.delenv("CARMA_MULTI_HESSIAN_BUDGET")
        for key in keys:
            np.testing.assert_array_equal(ch[key], full[key], err_msg="chunked " + key)
        # a subset of the curves in a multi-series of their own
        sub = [12, 3, 7, 0]
        ms = C.MultiSeries(np.concatenate([ts[c] for c in sub]), np.concatenate([ys[c] for c in sub]),
                           np.concatenate([es[c] for c in sub]), np.cumsum([0] + [len(ts[c]) for c in sub]))
        part = ms.hessian(kind, p, q, th[sub])
        ms.close()
        for key in keys:
            np.testing.assert_array_equal(part[key], full[key][sub], err_msg="subset " + key)
        # the single-curve form
        for c in (0, 5, 12):
            one = cp.CarmaModel(ts[c], ys[c], es[c], p=p, q=q).hessian(th[c])
            assert one.loglik == full.loglik[c] and one.status == full.status[c]
            for key in ("grad", "hessian", "cov", "stderr", "step"):
                np.testing.assert_array_equal(one[key], full[key][c], err_msg="CarmaModel %s %s" % (name, key))
    m.close()


def test_status_paths(C):
    m, ts, ys, es = _ragged_survey(C, seed=5)
    pri = m.default_priors()
    # REJECTED: sigma_y < 0 under flags 0
    name, kind, p, q, tail = _models(C)[2]
    th = _thetas(ys, tail, seed=1, bad=False)
    th[3, 0] = -0.5
    r = m.hessian(kind, p, q, th, flags=0)
    assert r.status[3] == C.HESS_REJECTED and r.loglik[3] == -np.inf
    assert np.all(np.isnan(r.grad[3])) and np.all(np.isnan(r.hessian[3])) and np.all(np.isnan(r.stderr[3]))
    # NOT_NEGDEF: sigma_y = 100 std(y) on a p >= 2 model under the default IGNORE_BOUNDS flags (under flags 0 it would
    # exceed max_stdev and come back REJECTED): there d^2 log p / d sigma^2 = n / sigma^2 - 3 r^2 / sigma^4 > 0
    th = _thetas(ys, tail, seed=1, bad=False)
    th[5, 0] = 100.0 * np.std(ys[5])
    r = m.hessian(kind, p, q, th)
    assert r.status[5] == C.HESS_NOT_NEGDEF and r.hessian[5, 0, 0] > 0
    assert np.all(np.isfinite(r.grad[5])) and np.all(np.isfinite(r.hessian[5]))
    assert np.all(np.isnan(r.cov[5])) and np.all(np.isnan(r.stderr[5]))
    assert m.hessian(kind, p, q, th, flags=0).status[5] == C.HESS_REJECTED
    # NONFINITE: a CAR(1) row on its prior's frequency bound (theta + h leaves it)
    name, kind, p, q, tail = _models(C)[0]
    th = _thetas(ys, tail, seed=2, bad=False)
    th[6, 3] = np.log(pri[6]["max_freq"]) - 2.0 ** -14
    r = m.hessian(kind, p, q, th)
    assert r.status[6] == C.HESS_NONFINITE and np.isfinite(r.loglik[6])
    assert np.all(np.isnan(r.grad[6])) and np.all(np.isnan(r.hessian[6])) and np.all(np.isnan(r.cov[6]))
    ok = np.arange(m.ncurves) != 6
    assert np.all(r.status[ok] != C.HESS_NONFINITE)
    m.close()


CALIBRATION = [   # (name, p, q, theta_true, ncurves, ny)
    ("car1", 1, 0, [1.0, 1.0, 0.0, np.log(1.0 / 3.0)], 3000, 1000),
    ("car2", 2, 0, None, 3000, 600),
]


@pytest.mark.parametrize("case", range(len(CALIBRATION)))
def test_laplace_widths_are_calibrated_at_the_fits(C, case):
    from carma_pack_b200 import synth
    name, p, q, truth, nc, ny = CALIBRATION[case]
    if truth is None:
        truth = [1.0, 1.0, 0.0] + list(synth.roots_to_logquad(np.array([-0.1 + 0.6j, -0.1 - 0.6j])))
    truth = np.array(truth)
    kind = C.KIND_CAR1 if p == 1 else C.KIND_CARP
    m = C.MultiSeries.simulate(nc, ny, kind, p, q, truth, yerr=0.05, dt_min=0.05, dt_max=20.0, seed=31 + case)
    fit = m.get_mle(p, q, ntrials=8, seed=7)
    r = m.hessian(kind, p, q, fit.x)
    np.testing.assert_array_equal(r.loglik, -fit.fun)
    d = truth.size
    on_box = np.zeros(nc, bool)
    cols = [j for j in range(d) if j != 1]            # measerr_scale: the box [0.9, 1.1] pins it
    for j in cols:
        w = fit.upper[:, j] - fit.lower[:, j]
        on_box |= np.isfinite(w) & ((fit.x[:, j] - fit.lower[:, j] < 1e-6 * w) | (fit.upper[:, j] - fit.x[:, j] < 1e-6 * w))
    keep = (r.status == C.HESS_OK) & ~on_box
    assert keep.mean() >= 0.9, (name, keep.mean(), np.bincount(r.status))
    z = (fit.x[keep][:, cols] - truth[cols]) / r.stderr[keep][:, cols]
    mean, sd = z.mean(axis=0), z.std(axis=0)
    gz = np.abs(r.grad[keep][:, cols]) * r.stderr[keep][:, cols]
    assert np.all(np.abs(mean) <= 0.15) and np.all((sd >= 0.85) & (sd <= 1.15)), (name, mean, sd)
    assert gz.max() <= GRAD_AT_FIT, (name, np.quantile(gz, [0.5, 0.99, 1.0]))
    m.close()
