"""In-tree build of the native pieces (sm_100a only):

  carma_pack_b200/libcarma_b200.so   CUDA kernels + the C ABI of include/carma_b200.h   (nvcc)
  carma_pack_b200/_carmcmc*.so       pybind11 module re-exporting the reference's `_carmcmc`
                                     surface on top of the C ABI                         (g++)

Run as  `python build_native.py [--force] [-v]`  or through  __graft_entry__.build().  Lives outside the
package on purpose: importing carma_pack_b200 loads libcarma_b200.so and must fail loudly when it is
missing, so the thing that creates the library cannot be inside it.
"""
import os
import shutil
import subprocess
import sys
import sysconfig

ROOT = os.path.dirname(os.path.abspath(__file__))
HERE = os.path.join(ROOT, "carma_pack_b200")
CSRC = os.path.join(HERE, "csrc")

NVCC = os.environ.get("NVCC") or shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
CXX = os.environ.get("CXX_HOST") or shutil.which("g++") or "g++"

CUDA_SOURCES = ["loglik.cu", "mcmc.cu", "scan.cu", "sim.cu", "mle.cu", "mle_dev.cu", "comm.cu", "survey.cu", "posterior.cu"]
CUDA_HEADERS = ["device_math.cuh", "fast_math.cuh", "theta_transform.cuh", "kalman_real.cuh", "kalman_cplx.cuh", "series.h",
                "hessian.cuh", "laplace.cuh", "select.cuh", os.path.join(ROOT, "include", "carma_b200.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr", "-Xptxas", "-v"]

LIB = os.path.join(HERE, "libcarma_b200.so")


def _newer(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def _run(cmd, log=None):
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if log:
        with open(log, "w") as f:
            f.write(" ".join(cmd) + "\n" + res.stdout)
    if res.returncode != 0:
        sys.stderr.write(res.stdout)
        raise RuntimeError("build failed: " + " ".join(cmd))
    return res.stdout


def build_cuda(force=False, verbose=False):
    srcs = [os.path.join(CSRC, s) for s in CUDA_SOURCES if os.path.exists(os.path.join(CSRC, s))]
    deps = srcs + [h if os.path.isabs(h) else os.path.join(CSRC, h) for h in CUDA_HEADERS]
    if not force and not _newer(LIB, deps):
        return LIB
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    from concurrent.futures import ThreadPoolExecutor

    def compile_one(src):
        o = os.path.join(HERE, "build", os.path.basename(src) + ".o")
        if not force and not _newer(o, [src] + deps[len(srcs):]):
            return o, ""
        return o, _run([NVCC] + NVCC_FLAGS + ["-c", src, "-o", o], log=o + ".log")

    with ThreadPoolExecutor(max_workers=len(srcs)) as ex:
        results = list(ex.map(compile_one, srcs))
    objs = [o for o, _ in results]
    if verbose:
        for _, out in results:
            print(out)
    _run([NVCC, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB] + objs + ["-cudart", "static", "-ldl"])
    return LIB


def pybind_module_path():
    suffix = sysconfig.get_config_var("EXT_SUFFIX") or ".so"
    return os.path.join(HERE, "_carmcmc" + suffix)


def build_pybind(force=False):
    src = os.path.join(CSRC, "host", "pymodule.cpp")
    if not os.path.exists(src):
        return None
    import pybind11
    out = pybind_module_path()
    host_dir = os.path.join(CSRC, "host")
    deps = [os.path.join(host_dir, f) for f in os.listdir(host_dir)] + [LIB]
    if not force and not _newer(out, deps):
        return out
    srcs = [os.path.join(host_dir, f) for f in sorted(os.listdir(host_dir)) if f.endswith(".cpp")]
    cmd = [CXX, "-O2", "-std=c++17", "-shared", "-fPIC", "-fvisibility=hidden",
           "-I" + pybind11.get_include(), "-I" + sysconfig.get_paths()["include"],
           "-I" + os.path.join(ROOT, "include"), "-I" + host_dir] + srcs + \
          ["-L" + HERE, "-lcarma_b200", "-Wl,-rpath,$ORIGIN", "-o", out]
    _run(cmd)
    return out


def build_all(force=False, verbose=False):
    lib = build_cuda(force=force, verbose=verbose)
    mod = build_pybind(force=force)
    return lib, mod


if __name__ == "__main__":
    print(build_all(force="--force" in sys.argv, verbose="-v" in sys.argv))
