"""CPU-side checks of carma_multi_simulate / MultiSeries.conditional_simulate: the entry point rejects a null handle,
null arrays and time offsets that do not start at 0 with CARMA_ERR_ARG and a message naming it, before any CUDA call;
the binding is declared.  The checks that need a multi-series (decreasing offsets, non-finite times, theta_rows,
curve_offset) are in tests/test_gpu_survey_simulate.py::test_argument_checks."""
import numpy as np
import pytest

CARMA_ERR_ARG = 1


def test_survey_simulate_rejects_bad_arguments_before_cuda():
    import carma_pack_b200 as C
    L = C._lib.lib
    th = np.zeros(8)
    so = np.array([0, 2, 3], dtype=np.int64)
    ts = np.zeros(3)
    out = np.zeros(16)

    def call(m=None, theta=th.ctypes.data, offs=so.ctypes.data, t=ts.ctypes.data, y=out.ctypes.data, npaths=2):
        return L.carma_multi_simulate(m, C.KIND_CARMA, 3, 1, None, theta, 2, 0, offs, t, npaths, 1, 0, y)

    for kw in ({}, {"theta": None}, {"offs": None}, {"t": None}, {"y": None}, {"npaths": 0}):
        assert call(**kw) == CARMA_ERR_ARG
        assert b"carma_multi_simulate" in L.carma_last_error() and b"null" in L.carma_last_error()
    bad = np.array([1, 2, 3], dtype=np.int64)
    assert call(offs=bad.ctypes.data) == CARMA_ERR_ARG
    assert b"carma_multi_simulate" in L.carma_last_error() and b"s_offsets" in L.carma_last_error()


def test_survey_simulate_binding_is_declared():
    import carma_pack_b200 as C
    assert "carma_multi_simulate" in C._lib.EXPORTED_SYMBOLS
    assert C._lib.lib.carma_multi_simulate.argtypes is not None
    assert callable(C.MultiSeries.conditional_simulate)


def test_conditional_simulate_shape_errors_raise_value_error():
    """The shape checks run before the handle is used, so an object without one shows them."""
    import carma_pack_b200 as C
    fake = object.__new__(C.MultiSeries)
    fake.ncurves = 2
    fake.offsets = np.array([0, 3, 6], dtype=np.int64)
    fake.handle = None
    d = C._lib.model_dim(C.KIND_CARMA, 3, 1)
    th = np.zeros((2, d))
    tq = np.arange(4.0)
    with pytest.raises(ValueError, match="theta"):
        fake.conditional_simulate(C.KIND_CARMA, 3, 1, np.zeros((3, d)), tq, [0, 2, 4])
    with pytest.raises(ValueError, match="theta"):
        fake.conditional_simulate(C.KIND_CARMA, 3, 1, np.zeros((2, 3, d)), tq, [0, 2, 4], npaths=2)
    with pytest.raises(ValueError, match="s_offsets"):
        fake.conditional_simulate(C.KIND_CARMA, 3, 1, th, tq, [0, 2])
    with pytest.raises(ValueError, match="s_offsets"):
        fake.conditional_simulate(C.KIND_CARMA, 3, 1, th, tq, [0, 2, 5])
    with pytest.raises(ValueError, match="npaths"):
        fake.conditional_simulate(C.KIND_CARMA, 3, 1, th, tq, [0, 2, 4], npaths=0)
