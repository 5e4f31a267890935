"""CPU-side checks of carma_psd_quantiles / carma_effective_samples and SurveySample: argument rejection before any CUDA
call, CARMA_ERR_CUDA without a device, the ctypes signatures, and the host-side summaries of SurveySample on injected
arrays (no device call)."""
import ctypes

import numpy as np
import pytest

CARMA_ERR_ARG, CARMA_ERR_CUDA = 1, 2


def _psd_call(C, kind=None, p=3, q=1, priors=None, nc=2, ns=4, theta=True, freq=True, rows=1, nf=3, pct=(16.0, 84.0),
              out=True):
    L = C._lib.lib
    kind = C.KIND_CARMA if kind is None else kind
    th = np.zeros(max(nc * ns * 17, 1))
    fr = np.ones(max(nc * nf, 1))
    pc = np.asarray(pct, dtype=float)
    o = np.zeros(max(nc * max(pc.size, 1) * nf, 1))
    return L.carma_psd_quantiles(kind, p, q, priors, nc, ns, th.ctypes.data if theta else None,
                                 fr.ctypes.data if freq else None, rows, nf, pc.ctypes.data if pc.size else None,
                                 pc.size, o.ctypes.data if out else None, None, 0)


def test_psd_quantiles_rejects_bad_arguments(C_host):
    C = C_host
    L = C._lib.lib
    bad = [dict(p=3, q=3), dict(p=8, q=0), dict(kind=C.KIND_CAR1, p=2, q=0), dict(kind=9),
           dict(pct=(50.0, 100.5)), dict(pct=(-1e-9,)), dict(pct=(float("nan"),)),
           dict(rows=3), dict(rows=0), dict(theta=False), dict(freq=False), dict(out=False),
           dict(kind=C.KIND_ZCARMA, p=3, q=0)]
    for kw in bad:
        assert _psd_call(C, **kw) == CARMA_ERR_ARG, kw
        assert b"carma_psd_quantiles" in L.carma_last_error()
    for kw in (dict(nc=0, theta=False, freq=False, out=False), dict(ns=0), dict(nf=0), dict(pct=())):
        assert _psd_call(C, **kw) == 0, kw
    # freq_rows = ncurves is accepted as well as 1
    assert _psd_call(C, rows=2, pct=(101.0,)) == CARMA_ERR_ARG and b"[0, 100]" in L.carma_last_error()


def test_effective_samples_rejects_null_and_skips_empty(C_host):
    L = C_host._lib.lib
    x, e = np.zeros(6), np.zeros(2)
    assert L.carma_effective_samples(1, 3, 2, None, e.ctypes.data, 0) == CARMA_ERR_ARG
    assert L.carma_effective_samples(1, 3, 2, x.ctypes.data, None, 0) == CARMA_ERR_ARG
    assert b"carma_effective_samples" in L.carma_last_error()
    assert L.carma_effective_samples(0, 3, 2, None, None, 0) == 0
    assert L.carma_effective_samples(1, 0, 2, None, None, 0) == 0


def test_no_device_gives_cuda_error(C_host):
    C = C_host
    if C._lib.device_count() > 0:
        pytest.skip("a CUDA device is visible: the no-device error path is checked on machines without one")
    assert _psd_call(C) == CARMA_ERR_CUDA
    x, e = np.zeros(6), np.zeros(2)
    assert C._lib.lib.carma_effective_samples(1, 3, 2, x.ctypes.data, e.ctypes.data, 0) == CARMA_ERR_CUDA


def test_bindings_are_declared(C_host):
    C = C_host
    L = C._lib.lib
    for name in ("carma_psd_quantiles", "carma_psd_quantiles_dev", "carma_effective_samples", "carma_effective_samples_dev"):
        assert name in C._lib.EXPORTED_SYMBOLS
    sz = ctypes.c_size_t
    assert L.carma_psd_quantiles.argtypes[4:6] == [sz, sz] and L.carma_psd_quantiles.argtypes[-1] is ctypes.c_int
    assert len(L.carma_psd_quantiles.argtypes) == 15 and len(L.carma_psd_quantiles_dev.argtypes) == 15
    assert L.carma_effective_samples.argtypes[:3] == [sz, sz, sz] and len(L.carma_effective_samples.argtypes) == 6
    assert len(L.carma_effective_samples_dev.argtypes) == 6
    assert callable(C.MultiSeries.run_mcmc)


def test_python_shape_checks(C_host):
    C = C_host
    with pytest.raises(ValueError, match="theta"):
        C._lib.psd_quantiles(C.KIND_CARMA, 3, 1, np.zeros((2, 5, 6)), np.ones(3), [50.0])
    with pytest.raises(ValueError, match="freq"):
        C._lib.psd_quantiles(C.KIND_CARMA, 3, 1, np.zeros((2, 5, 7)), np.ones((3, 3)), [50.0])
    with pytest.raises(ValueError, match="priors"):
        C._lib.psd_quantiles(C.KIND_ZCARMA, 3, 0, np.zeros((2, 5, 7)), np.ones(3), [50.0],
                             priors=np.zeros(3, dtype=C._lib.PRIOR_DTYPE))
    with pytest.raises(ValueError, match="x must be"):
        C._lib.effective_samples(np.zeros((4, 3)))


def _injected(C, nc=4, ns=300, seed=0):
    rng = np.random.default_rng(seed)
    trace = rng.normal(size=(nc, ns, 7))
    trace[:, :, 1] = rng.uniform(0.9, 1.1, (nc, ns))
    logpost = rng.normal(-100.0, 3.0, (nc, ns))
    stats = np.zeros(nc, dtype=C._lib.CURVE_STATS_DTYPE)
    stats["tspan"] = 100.0 + 10.0 * np.arange(nc)
    stats["min_dt"] = 0.05 + 0.01 * np.arange(nc)
    return C.SurveySample(trace, logpost, 3, 1, stats=stats), trace, logpost, stats


def test_surveysample_host_summaries_match_carmasample(C_host):
    C = C_host
    ss, trace, logpost, stats = _injected(C)
    best, dic, th_map = ss.best_index(), ss.DIC(), ss.map_theta()
    assert best.shape == (4,) and dic.shape == (4,) and th_map.shape == (4, 7)
    for c in range(4):
        cs = C.CarmaSample(np.arange(5.0), np.zeros(5), np.ones(5), trace=trace[c], logpost=logpost[c], p=3, q=1,
                           postprocess="numpy")
        assert best[c] == cs.best_index()
        assert dic[c] == cs.DIC()
        np.testing.assert_array_equal(th_map[c], trace[c, cs.best_index()])
        for name in ("var", "mu", "measerr_scale", "quad_coefs", "loglik", "loglik_only"):
            np.testing.assert_array_equal(ss.get_samples(name)[c], cs.get_samples(name).reshape(ss.get_samples(name)[c].shape))
    fr = ss.default_freq()
    assert fr.shape == (4, 200)
    for c in range(4):
        want = np.logspace(np.log10(1.0 / stats["tspan"][c]), np.log10(0.5 / stats["min_dt"][c]), 200)
        np.testing.assert_array_equal(fr[c], want)
    with pytest.raises(KeyError):
        ss.get_samples("log_omega")


def test_surveysample_car1_names(C_host):
    C = C_host
    rng = np.random.default_rng(2)
    trace = rng.normal(size=(3, 50, 4))
    trace[:, :, 1] = rng.uniform(0.9, 1.1, (3, 50))
    logpost = rng.normal(size=(3, 50))
    ss = C.SurveySample(trace, logpost, 1, 0)
    for c in range(3):
        cs = C.Car1Sample(np.arange(5.0), np.zeros(5), np.ones(5), trace=trace[c], logpost=logpost[c])
        for name in ("sigma", "log_omega", "var", "loglik_only"):
            np.testing.assert_array_equal(ss.get_samples(name)[c], np.ravel(cs.get_samples(name)))
    with pytest.raises(ValueError):
        C.SurveySample(trace, logpost[:, :10], 1, 0)
    with pytest.raises(ValueError):
        C.SurveySample(trace, logpost, 3, 1)


@pytest.fixture(scope="module")
def C_host():
    import carma_pack_b200 as c
    return c
