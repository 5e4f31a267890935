"""Survey-scale posterior summaries (carma_psd_quantiles, carma_effective_samples, MultiSeries.run_mcmc, SurveySample).

  * every percentile of the band is bitwise np.percentile of the kernel's own PSD values, on both selection paths,
    and the two paths agree bit for bit;
  * the PSD values equal a host evaluation of the same formula from carma_derived_params, and the polynomial form of
    CarmaSample.psd_credible_band / power_spectrum to rounding;
  * an output depends only on its curve: subsets, freq_rows and chunking change no bit; NaN rows poison only their curve;
  * the ESS kernel is MCMCSample.effective_samples;
  * SurveySample is CarmaSample per curve, and MultiSeries.run_mcmc is CarmaModel.run_mcmc per curve;
  * carma_derived_params returns what it returned before its body became the shared derive_row helper."""
import hashlib

import numpy as np
import pytest

from test_gpu_survey_filter import _models

pytestmark = pytest.mark.gpu

PCTS = [0.0, 2.5, 16.0, 50.0, 84.0, 97.5, 100.0]
TWO_PI = 2.0 * np.pi


@pytest.fixture(scope="module")
def C():
    import carma_pack_b200 as c
    if c._lib.device_count() < 1:
        pytest.fail("no CUDA device visible: GPU tests must run on the B200 box")
    return c


def _zpriors(C, nc):
    """Per-curve priors with different kappa bounds (the only fields the PSD kernels read)."""
    pri = np.zeros(nc, dtype=C._lib.PRIOR_DTYPE)
    pri["max_stdev"], pri["max_freq"], pri["min_freq"], pri["measerr_dof"] = 10.0, 10.0, 1e-4, 50.0
    pri["kappa_low"] = 0.2 + 0.1 * np.arange(nc)
    pri["kappa_high"] = 3.0 + 0.5 * np.arange(nc)
    return pri


def _trace(C, model, nc, ns, seed, scatter=0.05):
    """(ncurves, nsamples, d) theta rows around the model's tail, and the priors the kind needs."""
    name, kind, p, q, tail = _models(C)[model]
    rng = np.random.default_rng(seed)
    d = C.model_dim(kind, p, q)
    th = np.empty((nc, ns, d))
    th[:, :, 0] = rng.uniform(0.5, 2.0, (nc, ns))
    th[:, :, 1] = rng.uniform(0.9, 1.2, (nc, ns))
    th[:, :, 2] = rng.normal(0.0, 1.0, (nc, ns))
    th[:, :, 3:] = np.asarray(tail) + rng.normal(0.0, scatter, (nc, ns, len(tail)))
    pri = _zpriors(C, nc) if kind == C.KIND_ZCARMA else None
    return name, kind, p, q, th, pri


def _freq(nf=37, lo=1e-3, hi=2.0):
    return np.logspace(np.log10(lo), np.log10(hi), nf)


def _host_psd(C, kind, p, q, th, freq, prior):
    """The kernel's formula evaluated in numpy from carma_derived_params output, one IEEE operation at a time."""
    der = C._lib.derived_params(kind, p, q, th, prior=prior)
    w, beta, sig = der["ar_roots"], der["ma_coefs"], der["sigma"]
    nb = q if kind == C.KIND_CARMA else (p - 1 if kind == C.KIND_ZCARMA else 0)
    om = TWO_PI * freq[None, :]
    nr = np.broadcast_to(beta[:, nb:nb + 1], (th.shape[0], freq.size)).copy()
    ni = np.zeros_like(nr)
    for k in range(nb - 1, -1, -1):
        r = beta[:, k:k + 1] - ni * om
        ni = nr * om
        nr = r
    num = nr * nr + ni * ni
    den = np.ones_like(num)
    for k in range(p):
        dr = -w[:, k:k + 1].real
        di = om - w[:, k:k + 1].imag
        den = den * (dr * dr + di * di)
    with np.errstate(all="ignore"):
        return (sig[:, None] * sig[:, None] * num) / den


def _prior_struct(C, pri, c):
    return None if pri is None else C.Prior(*[float(v) for v in pri[c]])


@pytest.mark.parametrize("ns", [1, 2, 7, 1000])
def test_band_is_bitwise_np_percentile_on_both_paths(C, monkeypatch, ns):
    for model in (0, 2, 6):
        name, kind, p, q, th, pri = _trace(C, model, 3, ns, seed=ns + model)
        fr = _freq()
        out, psd = C._lib.psd_quantiles(kind, p, q, th, fr, PCTS, priors=pri, return_psd=True)
        want = np.percentile(psd, PCTS, axis=1).transpose(1, 0, 2)
        np.testing.assert_array_equal(out, want, err_msg="%s ns=%d" % (name, ns))
        assert np.all(np.isfinite(out))
        monkeypatch.setenv("CARMA_PSD_GLOBAL_SELECT", "1")
        out_g, psd_g = C._lib.psd_quantiles(kind, p, q, th, fr, PCTS, priors=pri, return_psd=True)
        monkeypatch.delenv("CARMA_PSD_GLOBAL_SELECT")
        np.testing.assert_array_equal(psd_g, psd, err_msg=name)
        np.testing.assert_array_equal(out_g, out, err_msg=name)


def test_ties_and_percentile_edges_follow_numpy(C, monkeypatch):
    """Repeated rows (equal PSD values around the selected order statistics) and percentiles just off the grid."""
    name, kind, p, q, th, pri = _trace(C, 2, 2, 50, seed=3)
    th[:, 10:30] = th[:, 10:11]
    pct = [0.0, 1e-9, 33.3, 49.999999, 50.0, 50.000001, 99.9999, 100.0]
    for env in (None, "1"):
        if env:
            monkeypatch.setenv("CARMA_PSD_GLOBAL_SELECT", env)
        out, psd = C._lib.psd_quantiles(kind, p, q, th, _freq(11), pct, return_psd=True)
        np.testing.assert_array_equal(out, np.percentile(psd, pct, axis=1).transpose(1, 0, 2))


@pytest.mark.parametrize("model", range(7))
def test_psd_values_match_root_and_polynomial_forms(C, model):
    from carma_pack_b200 import synth
    name, kind, p, q, th, pri = _trace(C, model, 3, 40, seed=100 + model)
    fr = _freq(53, 1e-4, 5.0)
    _, psd = C._lib.psd_quantiles(kind, p, q, th, fr, [50.0], priors=pri, return_psd=True)
    assert np.all(np.isfinite(psd)) and np.all(psd > 0)
    for c in range(th.shape[0]):
        host = _host_psd(C, kind, p, q, th[c], fr, _prior_struct(C, pri, c))
        np.testing.assert_allclose(psd[c], host, rtol=1e-12, atol=0, err_msg=name)
        der = C._lib.derived_params(kind, p, q, th[c], prior=_prior_struct(C, pri, c))
        for s in (0, 17, 39):
            ma = der["ma_coefs"][s] if kind == C.KIND_ZCARMA else der["ma_coefs"][s][:q + 1]
            poly = synth.power_spectrum(fr, der["sigma"][s], der["ar_coefs"][s], ma)
            np.testing.assert_allclose(psd[c, s], poly, rtol=1e-8, atol=0, err_msg="%s sample %d" % (name, s))
        if kind in (C.KIND_CARP, C.KIND_CARMA):
            cs = C.CarmaSample(np.arange(5.0), np.zeros(5), np.ones(5), trace=th[c], logpost=np.zeros(40), p=p, q=q)
            lo, hi, mid, _ = cs.psd_credible_band(percentile=68.0, nsamples=None, freq=fr)
            got = C._lib.psd_quantiles(kind, p, q, th[c:c + 1], fr, [16.0, 84.0, 50.0])[0]
            np.testing.assert_allclose(got, np.stack([lo, hi, mid]), rtol=1e-8, atol=0, err_msg=name)


def test_output_depends_only_on_its_curve(C, monkeypatch):
    name, kind, p, q, th, pri = _trace(C, 6, 9, 300, seed=7)
    rng = np.random.default_rng(1)
    fr1 = _freq(29)
    frn = np.sort(rng.uniform(1e-3, 3.0, (9, 29)), axis=1)
    for fr in (fr1, frn):
        full = C._lib.psd_quantiles(kind, p, q, th, fr, PCTS, priors=pri)
        sub = [1, 4, 8]
        part = C._lib.psd_quantiles(kind, p, q, th[sub], fr if fr.ndim == 1 else fr[sub], PCTS, priors=pri[sub])
        np.testing.assert_array_equal(part, full[sub])
        # each curve in a chunk of its own (the budget fits one curve)
        monkeypatch.setenv("CARMA_PSD_BUDGET", "1")
        chunked, psd = C._lib.psd_quantiles(kind, p, q, th, fr, PCTS, priors=pri, return_psd=True)
        monkeypatch.delenv("CARMA_PSD_BUDGET")
        np.testing.assert_array_equal(chunked, full)
        np.testing.assert_array_equal(chunked, np.percentile(psd, PCTS, axis=1).transpose(1, 0, 2))
    # freq_rows = ncurves with identical rows equals freq_rows = 1
    same = C._lib.psd_quantiles(kind, p, q, th, np.tile(fr1, (9, 1)), PCTS, priors=pri)
    np.testing.assert_array_equal(same, C._lib.psd_quantiles(kind, p, q, th, fr1, PCTS, priors=pri))


def test_large_survey_runs_in_several_chunks(C, monkeypatch):
    """4 GiB budget: 12 curves x 25,000 samples x 900 frequencies (with the PSD returned) need more than one chunk."""
    name, kind, p, q, th, pri = _trace(C, 2, 12, 25000, seed=5)
    fr = _freq(900)
    out, psd = C._lib.psd_quantiles(kind, p, q, th, fr, [16.0, 50.0, 84.0], return_psd=True)
    assert 12 * 25000 * 900 * 16 > 4 << 30
    np.testing.assert_array_equal(out, np.percentile(psd, [16.0, 50.0, 84.0], axis=1).transpose(1, 0, 2))
    sub = C._lib.psd_quantiles(kind, p, q, th[[0, 11]], fr, [16.0, 50.0, 84.0])
    np.testing.assert_array_equal(sub, out[[0, 11]])


def test_long_columns_are_exact_on_the_global_path(C):
    name, kind, p, q, th, pri = _trace(C, 4, 1, 41000, seed=9)
    out, psd = C._lib.psd_quantiles(kind, p, q, th, _freq(13), PCTS, return_psd=True)
    np.testing.assert_array_equal(out, np.percentile(psd, PCTS, axis=1).transpose(1, 0, 2))


def test_nan_rows_poison_only_their_curve(C, monkeypatch):
    name, kind, p, q, th, pri = _trace(C, 3, 4, 120, seed=11)
    th[1, 17, 3] = np.nan
    th[2, 5, 0] = np.inf
    for env in (None, "1"):
        if env:
            monkeypatch.setenv("CARMA_PSD_GLOBAL_SELECT", env)
        out, psd = C._lib.psd_quantiles(kind, p, q, th, _freq(), PCTS, return_psd=True)
        assert np.all(np.isnan(out[1])) and np.all(np.isnan(out[2]))
        assert np.all(np.isnan(psd[1, 17])) and np.all(np.isnan(psd[2, 5]))
        assert np.all(np.isfinite(out[[0, 3]]))
        np.testing.assert_array_equal(out, np.percentile(psd, PCTS, axis=1).transpose(1, 0, 2))


def _ar1(rng, phi, n, k):
    x = np.empty((n, k))
    x[0] = rng.standard_normal(k)
    for i in range(1, n):
        x[i] = phi * x[i - 1] + rng.standard_normal(k)
    return x


def test_ess_matches_mcmcsample(C):
    rng = np.random.default_rng(4)
    xs = [_ar1(rng, phi, 1000, 3) for phi in (0.0, 0.5, 0.9, 0.99)]
    const = np.full((1000, 3), 3.0)
    const[:, 1] = -0.5
    xs.append(const)
    x = np.stack(xs)
    ess = C._lib.effective_samples(x)
    for s in range(x.shape[0]):
        ms = C.MCMCSample()
        ms._samples["x"] = x[s]
        np.testing.assert_allclose(ess[s], ms.effective_samples("x"), rtol=1e-10, atol=0)
    np.testing.assert_array_equal(ess[-1], [1000.0] * 3)
    # a stuck chain at a value whose 1000-fold sum rounds: still ess = n (its residuals are zero)
    assert np.sum(np.full(1000, 0.1)) / 1000 != 0.1
    np.testing.assert_array_equal(C._lib.effective_samples(np.full((2, 1000, 2), 0.1)), np.full((2, 2), 1000.0))


@pytest.fixture(scope="module")
def survey(C):
    """Five CARMA(3,1) light curves of 150 to 400 points, times from 0, and their posterior samples (3 ensembles)."""
    from carma_pack_b200 import synth
    rng = np.random.default_rng(8)
    ar, ma, s2 = synth.carma31_truth()
    ts, ys, es, off = [], [], [], [0]
    for ny in (150, 400, 220, 310, 180):
        t = np.concatenate([[0.0], np.cumsum(rng.uniform(0.2, 3.0, ny - 1))])
        ts.append(t); ys.append(2.0 + synth.carma_process(t, s2, ar, ma, rng) + 0.2 * rng.standard_normal(ny))
        es.append(rng.uniform(0.1, 0.3, ny)); off.append(off[-1] + ny)
    m = C.MultiSeries(np.concatenate(ts), np.concatenate(ys), np.concatenate(es), off)
    return m, m.run_mcmc(3, 1, 120, n_ensembles=3, seed=77)


def test_surveysample_matches_carmasample_per_curve(C, survey):
    m, ss = survey
    assert ss.trace.shape == (5, 360, 7) and ss.logpost.shape == (5, 360)
    best, theta_map, dic = ss.best_index(), ss.map_theta(), ss.DIC()
    names = ["var", "mu", "measerr_scale", "quad_coefs", "ar_roots", "psd_width", "psd_centroid", "ar_coefs", "ma_coefs",
             "sigma", "loglik", "loglik_only"]
    got = {n: ss.get_samples(n) for n in names}
    ess = ss.effective_samples("sigma")
    lo, hi, mid, fr = ss.psd_credible_band()
    tq = np.linspace(-5.0, 250.0, 17)
    qm, qv = m.predict(C.KIND_CARMA, 3, 1, theta_map, np.tile(tq, 5), np.arange(6) * tq.size, priors=ss.priors)
    for c in range(5):
        cs = ss.curve(c)
        for n in names:
            np.testing.assert_array_equal(got[n][c], cs.get_samples(n).reshape(got[n][c].shape), err_msg=n)
        assert best[c] == cs.best_index() and dic[c] == cs.DIC()
        np.testing.assert_allclose(ess[c], cs.effective_samples("sigma"), rtol=1e-10, atol=0)
        t = m.curve(c)[0]
        want_fr = np.logspace(np.log10(1.0 / (t.max() - t.min())), np.log10(0.5 / np.diff(t).min()), 200)
        np.testing.assert_allclose(fr[c], want_fr, rtol=1e-13)
        wlo, whi, wmid, _ = cs.psd_credible_band(nsamples=None, freq=fr[c])
        for a, b in ((lo, wlo), (hi, whi), (mid, wmid)):
            np.testing.assert_allclose(a[c], b, rtol=1e-8, atol=0)
        pm, pv = cs.predict(tq)
        sl = slice(c * tq.size, (c + 1) * tq.size)
        scale = max(np.std(m.curve(c)[1]), 1.0)
        np.testing.assert_allclose(qm[sl], pm, rtol=0, atol=1e-6 * scale)
        np.testing.assert_allclose(qv[sl], pv, rtol=1e-6, atol=0)


def test_surveysample_ess_on_a_pt_run_trace(C, survey):
    m, ss = survey
    ess = ss.effective_samples("quad_coefs")
    for c in range(m.ncurves):
        np.testing.assert_allclose(ess[c], ss.curve(c).effective_samples("quad_coefs"), rtol=1e-10, atol=0)


@pytest.mark.parametrize("p,q", [(1, 0), (3, 1)])
def test_run_mcmc_curve0_equals_carmamodel(C, survey, p, q):
    m, _ = survey
    ss = m.run_mcmc(p, q, 60, n_ensembles=2, seed=5)
    t, y, e = m.curve(0)
    cs = C.CarmaModel(t, y, e, p, q).run_mcmc(60, seed=5, n_ensembles=2)
    np.testing.assert_array_equal(ss.trace[0], cs._trace)
    np.testing.assert_array_equal(ss.logpost[0], np.ravel(cs.get_samples("logpost")))
    np.testing.assert_array_equal(ss.get_samples("sigma")[0], np.ravel(cs.get_samples("sigma")))
    if p == 1:
        lo, hi, mid, fr = ss.psd_credible_band()
        assert np.all(np.isfinite(lo)) and np.all(lo <= mid) and np.all(mid <= hi)


# sha256 of carma_derived_params' output (float64 bytes) on 200,000 seeded rows per model, taken from the build before
# derived_params_kernel called derive_row
DERIVED_SHA256 = {
    "car1": "29c96f90d9f3ddedbfe1d5462887ccbdc8952794400582b27b084462a5c9cc74",
    "car2": "4fdb63b98b42cbb18db88c5379c0b122e278bbe96f04bb1f8996e8b163a91893",
    "carma31_conj": "971a98057d09d63273b1bb92cfb6100db7ab2d6caef636f428aab300aff724ba",
    "carma31_real": "bc97ed828d12dc8b9c9ca6af5b91bc9c82090670288bfef7f9e25877d25c45e3",
    "carma53": "8b8c19a19a401d6d55a83f7af554f187d4aa29849b254b23698d3e8e637f5b0e",
    "carma76": "5ee36703bda15db79b4d66a70329053a3591a9243bc2095a7ae2b46ab76dc95d",
    "zcarma5": "a48d17dfd7a275fb3b2a5bc2f0b40391fab6fb013724e9d96552d20438ba35d9",
}


def derived_digests(C, n=200000):
    out = {}
    prior = C.Prior(10.0, 10.0, 1e-4, 0.3, 4.0, 50.0)
    for model in range(7):
        name, kind, p, q, th, _ = _trace(C, model, 1, n, seed=1000 + model, scatter=0.5)
        th = th[0]
        th[::997, 0] = -1.0
        th[::1009, 3] = np.nan
        der = C._lib.derived_params(kind, p, q, th, prior=prior if kind == C.KIND_ZCARMA else None)
        h = hashlib.sha256()
        for key in ("ar_roots", "ar_coefs", "ma_coefs", "sigma", "psd_width", "psd_centroid"):
            h.update(np.ascontiguousarray(der[key]).tobytes())
        out[name] = h.hexdigest()
    return out


def test_derived_params_unchanged(C):
    assert derived_digests(C) == DERIVED_SHA256
