"""CPU-side checks of the survey-scale fits: the ctypes layout of carma_curve_stats_t, argument checks of
carma_multi_mle_grid_device before any CUDA call, and the box / redraw helpers that CarmaModel and MultiSeries share,
against a literal copy of the per-row loop they replaced."""
import ctypes
import os
import re

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_curve_stats_layout_matches_header():
    import carma_pack_b200 as C
    hdr = open(os.path.join(ROOT, "include", "carma_b200.h")).read()
    body = re.search(r"typedef struct carma_curve_stats \{(.*?)\} carma_curve_stats_t;", hdr, flags=re.S).group(1)
    fields = []
    for decl in body.split(";"):
        decl = decl.strip()
        if not decl:
            continue
        ctype, names = decl.split(None, 1)
        fields += [(n.strip(), ctype) for n in names.split(",")]
    cs = C._lib.CurveStats
    assert [n for n, _ in cs._fields_] == [n for n, _ in fields]
    sizes = {"double": 8, "int64_t": 8}
    off = 0
    for (name, ct), (pname, pct) in zip(fields, cs._fields_):
        assert getattr(cs, pname).offset == off and ctypes.sizeof(pct) == sizes[ct], name
        off += sizes[ct]
    assert ctypes.sizeof(cs) == off == 64
    assert C._lib.CURVE_STATS_DTYPE.itemsize == 64
    assert list(C._lib.CURVE_STATS_DTYPE.names) == [n for n, _ in fields]


def test_multi_grid_rejects_bad_arguments_before_cuda():
    import carma_pack_b200 as C
    L = C._lib.lib
    assert L.carma_multi_mle_grid_device(None, 0, None, None, None, None, None, None, None, None, None, None) != 0
    assert b"carma_multi_mle_grid_device" in L.carma_last_error()
    assert L.carma_multi_series_curve_stats(None, None) != 0
    assert b"carma_multi_series_curve_stats" in L.carma_last_error()


def _bounds_as_before(time, y, p, q):
    """CarmaModel._mle_bounds before it was shared with the survey path (literal copy)."""
    ysigma = y.std()
    dt = np.diff(time)
    max_freq = 0.9 / dt.min()
    min_freq = 1.0 / (time.max() - time.min())
    lo = [ysigma / 10.0, 0.9, -np.inf]
    hi = [10.0 * ysigma, 1.1, np.inf]
    if p == 1:
        lo.append(np.log(min_freq)); hi.append(np.log(max_freq))
    else:
        lo += [np.log(min(min_freq ** 2, 2.0 * min_freq))] * p
        hi += [np.log(max(max_freq ** 2, 2.0 * max_freq))] * p
        lo += [-np.inf] * q
        hi += [np.inf] * q
    return np.array(lo), np.array(hi)


def _redraw_as_before(x0, lo, hi, seed, trial_offset):
    """The out-of-box redraw of CarmaModel.mle_starts before it was shared (literal copy)."""
    ntrials, d = x0.shape
    for i in range(ntrials):
        rng = np.random.default_rng([seed % (2 ** 63), trial_offset + i])
        for j in range(d):
            if np.isfinite(lo[j]) and ((x0[i, j] < lo[j]) or (x0[i, j] > hi[j])):
                x0[i, j] = rng.uniform(lo[j], hi[j])
    return x0


def test_shared_box_and_redraw_equal_the_per_row_loop_bitwise():
    from carma_pack_b200.carma_pack import CarmaModel, mle_bounds, redraw_out_of_box
    rng = np.random.default_rng(2024)
    for trial in range(12):
        ny = int(rng.integers(5, 300))
        t = np.cumsum(rng.exponential(rng.uniform(0.1, 5.0), ny)) + rng.uniform(-100, 100)
        y = rng.normal(rng.uniform(-5, 5), rng.uniform(0.01, 10.0), ny)
        for p, q in ((1, 0), (2, 0), (3, 1), (5, 2), (7, 6)):
            lo0, hi0 = _bounds_as_before(t, y, p, q)
            model = CarmaModel(t, y, np.ones(ny))
            lo1, hi1 = model._mle_bounds(p, q)
            np.testing.assert_array_equal(lo1, lo0)
            np.testing.assert_array_equal(hi1, hi0)
            # the survey form: many curves' statistics at once, row c equal to curve c's box
            lo2, hi2 = mle_bounds(p, q, np.array([y.std(), 2.0]), np.array([np.diff(t).min(), 0.5]),
                                  np.array([t.max() - t.min(), 99.0]))
            np.testing.assert_array_equal(lo2[0], lo0)
            np.testing.assert_array_equal(hi2[0], hi0)
            d = lo0.size
            # starts partly outside the box (and a NaN, which neither version touches)
            x0 = rng.normal(0.0, 3.0, (40, d)) * np.maximum(np.abs(np.nan_to_num(hi0, posinf=1.0)), 1.0)
            x0[3, -1] = np.nan
            seed = int(rng.integers(0, 2 ** 64, dtype=np.uint64))
            off = int(rng.integers(0, 10 ** 6))
            a = _redraw_as_before(x0.copy(), lo0, hi0, seed, off)
            b = redraw_out_of_box(x0.copy(), lo0, hi0, seed, off + np.arange(40))
            np.testing.assert_array_equal(a, b)
            # per-row boxes (the survey path): rows of two curves with their own boxes and trial numbers
            b2 = redraw_out_of_box(np.concatenate([x0, x0]), np.concatenate([np.tile(lo0, (40, 1)), np.tile(lo2[1], (40, 1))]),
                                   np.concatenate([np.tile(hi0, (40, 1)), np.tile(hi2[1], (40, 1))]), seed,
                                   np.concatenate([off + np.arange(40), 7 + np.arange(40)]))
            np.testing.assert_array_equal(b2[:40], a)
            np.testing.assert_array_equal(b2[40:], _redraw_as_before(x0.copy(), lo2[1], hi2[1], seed, 7))
