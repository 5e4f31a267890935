"""CPU-side checks of the drop-in boundary: the C-ABI library loads without a GPU, exports every
symbol declared in include/carma_b200.h, validates arguments, and fails loudly (never falls back to
a CPU path) when asked to compute without CUDA."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_functions():
    src = open(os.path.join(ROOT, "include", "carma_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(carma_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_all_exported():
    import carma_pack_b200 as C
    names = declared_functions()
    assert len(names) >= 20
    for n in names:
        assert hasattr(C._lib.lib, n), "libcarma_b200.so does not export %s" % n
    # and the python binding knows every one of them
    assert set(names) == set(C._lib.EXPORTED_SYMBOLS)
    assert C._lib.lib.carma_abi_version() == 5


def test_struct_layouts_match_header():
    import carma_pack_b200 as C
    assert ctypes.sizeof(C.Prior) == 6 * 8
    assert ctypes.sizeof(C.PTOpts) == 72
    assert C._lib.TRACE_DTYPE.itemsize == 40
    assert C._lib.PRIOR_DTYPE.itemsize == 48
    o = C.PTOpts()
    C._lib.lib.carma_pt_default_opts(ctypes.byref(o))
    # defaults of RunCarmaSampler: carmcmc.cpp:92, 139, 141; steps.cpp:29
    assert (o.tmax, o.dof, o.target_rate) == (100.0, 8, 0.25)
    assert abs(o.gamma - 2.0 / 3.0) < 1e-16 and o.ntemps == 10 and o.thin == 1
    assert ctypes.sizeof(C._lib.MLEOpts) == 4 * 4 + 3 * 8
    m = C._lib.MLEOpts()
    C._lib.lib.carma_mle_default_opts(ctypes.byref(m))
    # scipy L-BFGS-B defaults used by the reference's fits (minimize(..., method="L-BFGS-B") at carma_pack.py:250): pgtol 1e-5, factr*eps 2.2e-9, eps 1e-8
    assert (m.maxiter, m.history, m.max_backtrack) == (1000, 8, 25)
    assert (m.gtol, m.ftol, m.fd_eps) == (1e-5, 2.2e-9, 1e-8)
    # carma_mle_job_t: 3 ints + flags, the prior, size_t nstart; CARMA_MAX_DIM = 3 + 2 * CARMA_MAX_P
    assert ctypes.sizeof(C._lib.MLEJob) == 4 * 4 + 6 * 8 + 8 and C._lib.MLEJob.prior.offset == 16
    hdr = open(os.path.join(ROOT, "include", "carma_b200.h")).read()
    assert int(re.search(r"#define CARMA_MAX_P (\d+)", hdr).group(1)) * 2 + 3 == C._lib.MAX_DIM
    # argument checks of the grid fit come before any CUDA call
    assert C._lib.lib.carma_mle_grid_device(None, 0, None, None, None, None, None, None, None, None, None, 0) != 0
    assert b"carma_mle_grid_device" in C._lib.lib.carma_last_error()


def test_argument_validation_without_gpu():
    import carma_pack_b200 as C
    t = np.arange(10.0)
    with pytest.raises(C.CarmaError):  # unsorted times are rejected before any CUDA call
        C.Series(t[::-1].copy(), t, t)
    with pytest.raises(C.CarmaError):
        C.Series(t[:1], t[:1], t[:1])
    with pytest.raises(ValueError):
        C.Series(t, t[:5], t)


def test_log_prior_host_helper():
    import carma_pack_b200 as C
    pr = C.Prior(10.0, 1.0, 0.01, 0.05, 1.0, 50.0)
    th = np.array([1.0, 1.3, 0.0, -1.0, -2.0, 0.4])
    want = -0.5 * 50 / 1.3 - 26.0 * np.log(1.3)  # carpack.hpp:118-126
    assert abs(C._lib.log_prior(C.KIND_CARP, 2, th, pr) - want) < 1e-14
    wantz = want - 0.4 - 2 * np.log(1 + np.exp(-0.4))  # carpack.hpp:444-456, theta[p+3]
    assert abs(C._lib.log_prior(C.KIND_ZCARMA, 2, th, pr) - wantz) < 1e-14


def test_no_cpu_fallback():
    """Without a CUDA device every compute entry point must raise, not silently compute on the CPU.  Checked in a
    child process that is shown no device, so that the check also runs on a machine with a GPU."""
    code = ("import numpy as np, pytest\n"
            "import carma_pack_b200 as C\n"
            "assert C._lib.device_count() == 0\n"
            "t = np.arange(10.0)\n"
            "with pytest.raises(C.CarmaError):\n"
            "    C.Series(t, np.sin(t), np.ones(10))\n"
            "with pytest.raises(C.CarmaError):\n"
            "    C._lib.fp64_peak_tflops(0)\n")
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert out.returncode == 0, out.stderr[-2000:]


def test_product_never_imports_oracle():
    """The oracle is test infrastructure: nothing under carma_pack_b200/ may reference it."""
    pkg = os.path.join(ROOT, "carma_pack_b200")
    for dirpath, _, files in os.walk(pkg):
        if os.path.basename(dirpath) == "build":
            continue
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".hpp", ".cpp")):
                txt = open(os.path.join(dirpath, f)).read()
                assert "liboracle" not in txt and "from oracle" not in txt and "import oracle" not in txt, f
                assert "carma_oracle" not in txt, f


def test_reference_package_alias_imports_on_cpu():
    """`import carmcmc` (the reference's package name) resolves to this implementation without a GPU."""
    import carmcmc
    for name in ("vecD", "vecvecD", "vecC", "pairD", "CAR1", "CARp", "CARMA", "run_mcmc_car1", "run_mcmc_carma",
                 "KalmanFilter1", "KalmanFilterp", "CarmaModel", "CarmaSample", "Car1Sample", "power_spectrum",
                 "carma_variance", "carma_process", "get_ar_roots", "MCMCSample"):
        assert hasattr(carmcmc, name), name
    v = carmcmc.vecD()
    v.extend([1.0, 2.0])
    v.append(3.0)
    assert len(v) == 3 and list(v) == [1.0, 2.0, 3.0] and v[1] == 2.0
    c = carmcmc.vecC()
    c.append(1 + 2j)
    assert c[0] == 1 + 2j
    pr = carmcmc.pairD()
    pr.first, pr.second = 1.5, 2.5
    assert (pr.first, pr.second) == (1.5, 2.5)
