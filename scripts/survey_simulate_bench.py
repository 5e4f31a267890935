"""Survey-scale conditional simulation on one GPU (MultiSeries.conditional_simulate / carma_multi_simulate), against
what a user does without it -- a Python loop of Series(curve).simulate -- on a subset of the curves.

  * end to end (host arrays in and out, blocking call) on --curves CARMA(3,1) curves of --ny points at the true
    parameters, --nq query times per curve over [-10 %, +110 %] of each span, unsorted, for every npaths in --npaths;
    best of --reps calls after a warm-up;
  * the split into the prior-draw, forward and query kernels: device time of each kernel from torch.profiler (CUDA
    activities), in a separate call of the same size;
  * the Python loop over --subset curves with --loop-npaths paths each.
The card's name and power limit are read in the same run.

    python scripts/survey_simulate_bench.py [--curves 10000] [--ny 1000] [--nq 100] [--npaths 1,16,128] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

KERNELS = ("condsim_prior_kernel", "predict_forward_kernel", "predict_query_kernel")


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
    return {k: {"device_s": round(out[k], 5), "launches": launches[k]} for k in KERNELS}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--curves", type=int, default=10000)
    ap.add_argument("--ny", type=int, default=1000)
    ap.add_argument("--nq", type=int, default=100)
    ap.add_argument("--npaths", default="1,16,128")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--subset", type=int, default=200)
    ap.add_argument("--loop-npaths", type=int, default=16)
    ap.add_argument("--seed", type=int, default=23)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    import carma_pack_b200 as C
    from carma_pack_b200 import synth
    if C._lib.device_count() < 1 or not torch.cuda.is_available():
        raise SystemExit("no CUDA device visible")
    torch.cuda.init()
    p, q, kind = 3, 1, C.KIND_CARMA
    th = synth.carma31_theta()
    nc, ny, nq = args.curves, args.ny, args.nq
    m = C.MultiSeries.simulate(nc, ny, kind, p, q, th, yerr=0.2, dt_min=0.05, dt_max=60.0, seed=args.seed)
    span = m.curve_stats()["tspan"]
    rng = np.random.default_rng(1)
    tq = (rng.uniform(-0.1, 1.1, (nc, nq)) * span[:, None]).reshape(-1)
    qo = np.arange(nc + 1, dtype=np.int64) * nq
    theta = np.tile(th, (nc, 1))

    runs = {}
    for npaths in [int(x) for x in args.npaths.split(",")]:
        def call():
            return m.conditional_simulate(kind, p, q, theta, tq, qo, npaths=npaths, seed=5)
        first = call()   # warm-up: module load, scratch growth
        walls = []
        for _ in range(args.reps):
            t0 = time.perf_counter()
            out = call()
            walls.append(time.perf_counter() - t0)
        best = min(walls)
        runs[str(npaths)] = {
            "npaths": npaths, "wall_s": round(best, 4), "wall_s_per_rep": [round(w, 4) for w in walls],
            "curves_per_s": float("%.4g" % (nc / best)), "draws_per_s": float("%.4g" % (nc * nq * npaths / best)),
            "repeat_bitwise_equal": bool(np.array_equal(first, out)), "all_finite": bool(np.all(np.isfinite(out))),
            "kernels": kernel_split(call),
        }
        del first, out

    # what a user does today: one Series per curve, explicit parameters from the theta row
    nsub = min(args.subset, nc)
    der = C._lib.derived_params(kind, p, q, th[None, :])
    s2, roots, ma = der["sigma"][0] ** 2, der["ar_roots"][0], der["ma_coefs"][0]
    curves = [m.curve(c) for c in range(nsub)]
    t, y, e = curves[0]
    C.Series(t, y, e).simulate(s2, roots, ma, tq[:nq], measerr_scale=th[1], mu=th[2], seed=5, npaths=args.loop_npaths)
    t0 = time.perf_counter()
    for c, (t, y, e) in enumerate(curves):
        s = C.Series(t, y, e)
        s.simulate(s2, roots, ma, tq[qo[c]:qo[c + 1]], measerr_scale=th[1], mu=th[2], seed=5, npaths=args.loop_npaths)
        s.close()
    t_loop = time.perf_counter() - t0
    m.close()

    name, power = card()
    out = {
        "what": "MultiSeries.conditional_simulate, CARMA(3,1) at the true parameters, %d simulated curves of ny = %d, "
                "%d query times per curve" % (nc, ny, nq),
        "gpu": name, "power_limit": power,
        "survey": runs,
        "python_loop": {"curves": nsub, "npaths": args.loop_npaths, "wall_s": round(t_loop, 3),
                        "curves_per_s": round(nsub / t_loop, 2),
                        "what": "Series(curve).simulate(%d times, %d paths) per curve" % (nq, args.loop_npaths)},
    }
    print(json.dumps(out))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
