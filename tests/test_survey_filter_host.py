"""CPU-side checks of the survey filter / diagnostics / predict entry points: every one rejects a null handle, bad
query offsets and bad nlags with CARMA_ERR_ARG and a message naming it, before any CUDA call."""
import ctypes

import numpy as np

CARMA_ERR_ARG = 1


def test_survey_filter_entry_points_reject_bad_arguments_before_cuda():
    import carma_pack_b200 as C
    L = C._lib.lib
    th = np.zeros(8)
    buf = np.zeros(8)
    ptr = th.ctypes.data

    def last():
        return L.carma_last_error()

    assert L.carma_multi_filter(None, C.KIND_CARMA, 3, 1, None, ptr, 0, buf.ctypes.data, buf.ctypes.data, None) == CARMA_ERR_ARG
    assert b"carma_multi_filter" in last()
    assert L.carma_multi_filter_dev(None, C.KIND_CARMA, 3, 1, ptr, ptr, 0, ptr, ptr, None, None) == CARMA_ERR_ARG
    assert b"carma_multi_filter_dev" in last()

    out = np.zeros(64)
    assert L.carma_multi_assess_fit(None, C.KIND_CARMA, 3, 1, None, ptr, 0, 20, out.ctypes.data) == CARMA_ERR_ARG
    assert b"carma_multi_assess_fit" in last()
    for nlags in (0, -1):
        assert L.carma_multi_assess_fit(None, C.KIND_CARMA, 3, 1, None, ptr, 0, nlags, out.ctypes.data) == CARMA_ERR_ARG
        assert b"carma_multi_assess_fit" in last() and b"nlags" in last()

    qo = np.array([0, 2, 3], dtype=np.int64)
    tq = np.zeros(3)
    assert L.carma_multi_predict(None, C.KIND_CARMA, 3, 1, None, ptr, 0, qo.ctypes.data, tq.ctypes.data, buf.ctypes.data,
                                 buf.ctypes.data) == CARMA_ERR_ARG
    assert b"carma_multi_predict" in last()
    bad = np.array([1, 2, 3], dtype=np.int64)   # query offsets that do not start at 0
    assert L.carma_multi_predict(None, C.KIND_CARMA, 3, 1, None, ptr, 0, bad.ctypes.data, tq.ctypes.data, buf.ctypes.data,
                                 buf.ctypes.data) == CARMA_ERR_ARG
    assert b"carma_multi_predict" in last() and b"q_offsets" in last()


def test_survey_filter_bindings_are_declared():
    import carma_pack_b200 as C
    for name in ("carma_multi_filter_dev", "carma_multi_filter", "carma_multi_assess_fit", "carma_multi_predict"):
        assert name in C._lib.EXPORTED_SYMBOLS
        assert getattr(C._lib.lib, name).argtypes is not None
    assert C.MultiSeries._default_flags(1, None) == 0
    assert C.MultiSeries._default_flags(3, None) == C.IGNORE_BOUNDS
    assert C.MultiSeries._default_flags(3, 0) == 0
    assert isinstance(C._lib.lib.carma_multi_predict, ctypes._CFuncPtr)
