"""Survey-scale Kalman smoother on one GPU (MultiSeries.smooth / carma_multi_smooth) against the only way to get the same
numbers without it, MultiSeries.predict with the wanted times as queries.

  * data times: the smoothed process at every curve's own data times -- smooth without queries against predict with
    every data time as a query (O(ny^2 / 2) filter steps per curve);
  * grid: --grid query times per curve on a regular grid over its span -- smooth with queries (with and without the
    per-point outputs, points=False) against predict;
  * end to end (host arrays in and out, blocking call) on --curves CARMA(3,1) curves of --ny points at the true
    parameters, best of --reps calls after a warm-up; device time per kernel from torch.profiler (CUDA activities) in a
    separate call of the same size; the largest difference between the two answers.
The card's name and power limit are read in the same run.

    python scripts/survey_smooth_bench.py [--curves 10000] [--ny 1000] [--grid 1000] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

KERNELS = ("multi_smooth_kernel", "predict_forward_kernel", "predict_query_kernel")


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
    return {k: {"device_s": round(out[k], 5), "launches": launches[k]} for k in KERNELS if launches[k]}


def timed(call, reps):
    first = call()   # warm-up: module load, scratch growth
    walls = []
    for _ in range(reps):
        t0 = time.perf_counter()
        call()
        walls.append(time.perf_counter() - t0)
    return first, {"wall_s": round(min(walls), 4), "wall_s_per_rep": [round(w, 4) for w in walls],
                   "kernels": kernel_split(call)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--curves", type=int, default=10000)
    ap.add_argument("--ny", type=int, default=1000)
    ap.add_argument("--grid", type=int, default=1000)
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
    p, q, kind = 3, 1, C.KIND_CARMA
    th = synth.carma31_theta()
    nc, ny, ng = args.curves, args.ny, args.grid
    m = C.MultiSeries.simulate(nc, ny, kind, p, q, th, yerr=0.2, dt_min=0.05, dt_max=60.0, seed=args.seed)
    theta = np.tile(th, (nc, 1))
    tdata = np.concatenate([m.curve(c)[0] for c in range(nc)])   # the axes of simulated curves start at 0
    span = m.curve_stats()["tspan"]
    tgrid = (np.linspace(0.0, 1.0, ng)[None, :] * span[:, None]).reshape(-1)
    qgrid = np.arange(nc + 1, dtype=np.int64) * ng

    res = {}
    s, rs = timed(lambda: m.smooth(kind, p, q, theta), args.reps)
    pr, rp = timed(lambda: m.predict(kind, p, q, theta, tdata, m.offsets), args.reps)
    res["data_times"] = {
        "smooth": rs, "predict": rp, "speedup_end_to_end": round(rp["wall_s"] / rs["wall_s"], 2),
        "max_abs_mean_diff": float("%.3g" % np.max(np.abs(s.mean - pr[0]))),
        "max_rel_var_diff": float("%.3g" % np.max(np.abs(s.var - pr[1]) / th[0] ** 2)),
    }
    s, rs = timed(lambda: m.smooth(kind, p, q, theta, tq=tgrid, q_offsets=qgrid), args.reps)
    s2, rs2 = timed(lambda: m.smooth(kind, p, q, theta, tq=tgrid, q_offsets=qgrid, points=False), args.reps)
    pr, rp = timed(lambda: m.predict(kind, p, q, theta, tgrid, qgrid), args.reps)
    res["grid"] = {
        "smooth": rs, "smooth_points_false": rs2, "predict": rp,
        "speedup_end_to_end": round(rp["wall_s"] / rs["wall_s"], 2),
        "speedup_end_to_end_points_false": round(rp["wall_s"] / rs2["wall_s"], 2),
        "points_false_bitwise_equal": bool(np.array_equal(s.qmean, s2.qmean) and np.array_equal(s.qvar, s2.qvar)),
        "max_abs_mean_diff": float("%.3g" % np.max(np.abs(s.qmean - pr[0]))),
        "max_rel_var_diff": float("%.3g" % np.max(np.abs(s.qvar - pr[1]) / th[0] ** 2)),
    }
    m.close()

    name, power = card()
    out = {
        "what": "MultiSeries.smooth vs MultiSeries.predict, CARMA(3,1) at the true parameters, %d simulated curves of "
                "ny = %d: at the data times, and at %d grid times per curve" % (nc, ny, ng),
        "gpu": name, "power_limit": power, **res,
    }
    print(json.dumps(out))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
