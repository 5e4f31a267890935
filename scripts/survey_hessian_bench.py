"""Survey-scale fit uncertainties on one GPU (MultiSeries.hessian / carma_multi_hessian) against the way to get the same
numbers without it: d^2 + d + 1 calls of MultiSeries.loglik on the documented stencil rows, assembled in numpy.

  * sizes: --curves CARMA(3,1) curves, --curves-large CARMA(3,1) curves and --curves CARMA(5,3) curves, all of --ny
    simulated points, at the true parameters;
  * end to end (host arrays in and out, blocking call), best of --reps calls after a warm-up; device time of the
    evaluation and assembly kernels from torch.profiler (CUDA activities) in a separate call, and of one
    multi_loglik_kernel (K4) launch on the same curves, for the per-evaluation rate of each;
  * the baseline's Hessians against the call's, relative to max|H| per curve (the ceiling of the tests: 1e-12).
The card's name and power limit are read in the same run.

    python scripts/survey_hessian_bench.py [--curves 10000] [--curves-large 100000] [--ny 1000] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

KERNELS = ("multi_hessian_eval_kernel", "multi_hessian_assemble_kernel", "multi_loglik_kernel")


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        name, power = out[0].split(",")
        return name.strip(), power.strip()
    except Exception as e:  # noqa: BLE001
        return "unknown (%s)" % e, "unknown"


def kernel_split(fn):
    """Device time per kernel family of one call of fn, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
    out = {k: 0.0 for k in KERNELS}
    launches = {k: 0 for k in KERNELS}
    for ev in prof.events():
        if ev.device_type.name != "CUDA":
            continue
        for k in KERNELS:
            if k in ev.name:
                out[k] += (ev.time_range.end - ev.time_range.start) * 1e-6   # microseconds
                launches[k] += 1
    return {k: {"device_s": round(out[k], 6), "launches": launches[k]} for k in KERNELS if launches[k]}


def timed(call, reps):
    first = call()   # warm-up: module load, scratch growth
    walls = []
    for _ in range(reps):
        t0 = time.perf_counter()
        call()
        walls.append(time.perf_counter() - t0)
    return first, {"wall_s": round(min(walls), 4), "wall_s_per_rep": [round(w, 4) for w in walls]}


def stencil(theta, rel_step):
    """The documented stencil rows of every curve: (npts, nc, d), and the steps (nc, d)."""
    from carma_pack_b200._lib import hessian_steps
    nc, d = theta.shape
    h = hessian_steps(theta, rel_step)
    rows = [theta]
    for sgn in (1.0, -1.0):
        for i in range(d):
            r = theta.copy()
            r[:, i] = theta[:, i] + h[:, i] if sgn > 0 else theta[:, i] - h[:, i]
            rows.append(r)
    for i in range(d):
        for j in range(i + 1, d):
            rp, rm = theta.copy(), theta.copy()
            rp[:, i], rp[:, j] = theta[:, i] + h[:, i], theta[:, j] + h[:, j]
            rm[:, i], rm[:, j] = theta[:, i] - h[:, i], theta[:, j] - h[:, j]
            rows += [rp, rm]
    return np.array(rows), h


def assemble(f, h):
    """numpy assembly of every curve: f (npts, nc), h (nc, d) -> H (nc, d, d)."""
    d = h.shape[1]
    f0, fp, fm = f[0], f[1:1 + d].T, f[1 + d:1 + 2 * d].T
    H = np.empty((h.shape[0], d, d))
    for i in range(d):
        H[:, i, i] = (fp[:, i] - 2.0 * f0 + fm[:, i]) / (h[:, i] * h[:, i])
    r = 0
    for i in range(d):
        for j in range(i + 1, d):
            num = f[1 + 2 * d + 2 * r] - fp[:, i] - fp[:, j] + 2.0 * f0 - fm[:, i] - fm[:, j] + f[2 + 2 * d + 2 * r]
            H[:, i, j] = H[:, j, i] = num / (2.0 * h[:, i] * h[:, j])
            r += 1
    return H


def case(C, label, kind, p, q, th, nc, ny, reps, seed):
    m = C.MultiSeries.simulate(nc, ny, kind, p, q, th, yerr=0.2, dt_min=0.05, dt_max=60.0, seed=seed)
    theta = np.tile(th, (nc, 1))
    flags = 0 if p == 1 else C.IGNORE_BOUNDS
    d = th.size
    npts = d * d + d + 1
    r, rh = timed(lambda: m.hessian(kind, p, q, theta), reps)
    rh["kernels"] = kernel_split(lambda: m.hessian(kind, p, q, theta))
    k4 = kernel_split(lambda: m.loglik(kind, p, q, theta, flags=flags))["multi_loglik_kernel"]["device_s"]

    def by_hand():
        rows, h = stencil(theta, C.HESS_REL_STEP)
        f = np.stack([m.loglik(kind, p, q, np.ascontiguousarray(rows[k]), flags=flags) for k in range(npts)])
        return assemble(f, h)

    H, rb = timed(by_hand, max(1, reps - 1))
    ok = np.all(np.isfinite(r.hessian.reshape(nc, -1)), axis=1) & np.all(np.isfinite(H.reshape(nc, -1)), axis=1)
    rel = np.abs(r.hessian[ok] - H[ok]).max(axis=(1, 2)) / np.abs(H[ok]).max(axis=(1, 2))
    ev = rh["kernels"]["multi_hessian_eval_kernel"]["device_s"]
    bitwise = bool(np.array_equal(r.loglik, m.loglik(kind, p, q, theta, flags=flags)))
    m.close()
    return {
        "model": label, "curves": nc, "ny": ny, "d": d, "stencil_points": npts,
        "hessian": rh, "by_hand": rb, "speedup_end_to_end": round(rb["wall_s"] / rh["wall_s"], 2),
        "k4_one_launch_device_s": round(k4, 6),
        "eval_kernel_evaluations_per_s": float("%.3g" % (nc * npts / ev)),
        "k4_curve_evaluations_per_s": float("%.3g" % (nc / k4)),
        "eval_vs_k4_per_evaluation": round((nc * npts / ev) / (nc / k4), 2),
        "status_counts": {str(s): int(n) for s, n in zip(*np.unique(r.status, return_counts=True))},
        "max_rel_hessian_diff_vs_by_hand": float("%.3g" % rel.max()) if rel.size else None,
        "loglik_bitwise_k4": bitwise,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--curves", type=int, default=10000)
    ap.add_argument("--curves-large", type=int, default=100000)
    ap.add_argument("--ny", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--seed", type=int, default=29)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    import carma_pack_b200 as C
    from carma_pack_b200 import synth
    if C._lib.device_count() < 1 or not torch.cuda.is_available():
        raise SystemExit("no CUDA device visible")
    torch.cuda.init()
    name, power = card()
    th31 = synth.carma31_theta()
    th53 = np.array([1.0, 1.0, 0.0] + list(synth.roots_to_logquad(np.array([-0.05 + 0.3j, -0.05 - 0.3j, -0.2, -0.9, -0.4])))
                    + list(synth.roots_to_logquad(np.array([-1.5 + 0.5j, -1.5 - 0.5j, -3.0]))))
    cases = [("CARMA(3,1)", 3, 1, th31, args.curves), ("CARMA(3,1)", 3, 1, th31, args.curves_large),
             ("CARMA(5,3)", 5, 3, th53, args.curves)]
    res = []
    for label, p, q, th, nc in cases:
        res.append(case(C, label, C.KIND_CARMA, p, q, th, nc, args.ny, args.reps, args.seed))
        print(json.dumps(res[-1]), flush=True)
    out = {
        "what": "MultiSeries.hessian vs d^2 + d + 1 MultiSeries.loglik calls + numpy assembly, simulated curves at the "
                "true parameters",
        "gpu": name, "power_limit": power, "cases": res,
    }
    print(json.dumps(out))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
