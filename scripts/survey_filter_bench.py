"""Survey-scale Kalman filter, fit diagnostics and prediction on one GPU (MultiSeries.kalman_filter / filter_dev,
assess_fit_values, predict), against what a user does without them -- a Python loop of Series(curve).filter /
.predict -- on a subset of the curves.

  * filter kernel: CARMA(3,1) at the true parameters on every curve of a simulated survey, device pointers
    (carma_multi_filter_dev), timed with CUDA events over --reps launches, alternated in the same process with
    carma_multi_loglik_dev (K4) on the same survey and with the block-store and scalar-store variants; curves/s and the
    algorithmic HBM rate (24 B read + 16 B written per point);
  * assess_fit_values (nlags 20) and kalman_filter end to end (host arrays in and out, blocking calls);
  * predict end to end on --pcurves curves x --nq query times each;
  * the Python loop over --subset curves.
The card's name and power limit are read in the same run.

    python scripts/survey_filter_bench.py [--curves 100000] [--ny 1000] [--pcurves 10000] [--nq 100] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        name, power = out[0].split(",")
        return name.strip(), power.strip()
    except Exception as e:  # noqa: BLE001
        return "unknown (%s)" % e, "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--curves", type=int, default=100000)
    ap.add_argument("--ny", type=int, default=1000)
    ap.add_argument("--pcurves", type=int, default=10000)
    ap.add_argument("--nq", type=int, default=100)
    ap.add_argument("--subset", type=int, default=200)
    ap.add_argument("--reps", type=int, default=10, help="launches per timed window of the filter kernels")
    ap.add_argument("--rounds", type=int, default=3, help="alternations of the three filter kernels")
    ap.add_argument("--seed", type=int, default=23)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    import carma_pack_b200 as C
    from carma_pack_b200 import synth
    if C._lib.device_count() < 1 or not torch.cuda.is_available():
        raise SystemExit("no CUDA device visible")
    p, q, kind = 3, 1, C.KIND_CARMA
    th = synth.carma31_theta()
    sim = dict(yerr=0.2, dt_min=0.05, dt_max=60.0)
    nc, ny = args.curves, args.ny
    m = C.MultiSeries.simulate(nc, ny, kind, p, q, th, seed=args.seed, **sim)
    theta = np.tile(th, (nc, 1))
    dev = torch.device("cuda:0")
    d_th = torch.from_numpy(theta).to(dev)
    d_pr = torch.from_numpy(m.default_priors().view(np.float64).reshape(nc, 6).copy()).to(dev)
    total = nc * ny
    d_mean = torch.empty(total, dtype=torch.float64, device=dev)
    d_var = torch.empty(total, dtype=torch.float64, device=dev)
    d_ll = torch.empty(nc, dtype=torch.float64, device=dev)
    d_k4 = torch.empty(nc, dtype=torch.float64, device=dev)

    def run(variant):
        if variant == "k4":
            m.loglik_dev(kind, p, q, d_pr.data_ptr(), d_th.data_ptr(), d_k4.data_ptr(), flags=C.IGNORE_BOUNDS)
        else:
            os.environ["CARMA_MULTI_FILTER_STORES"] = variant
            m.filter_dev(kind, p, q, d_pr.data_ptr(), d_th.data_ptr(), d_mean.data_ptr(), d_var.data_ptr(),
                         d_ll.data_ptr())

    variants = ("block", "scalar", "k4")
    outputs = {}
    for v in variants:   # warm-up, and the outputs of each variant for the equality checks
        run(v)
        torch.cuda.synchronize()
        outputs[v] = (d_mean.cpu().numpy().copy(), d_var.cpu().numpy().copy(), d_ll.cpu().numpy().copy()) \
            if v != "k4" else d_k4.cpu().numpy().copy()
    times = {v: [] for v in variants}
    for _ in range(args.rounds):
        for v in variants:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.reps):
                run(v)
            e1.record()
            e1.synchronize()
            times[v].append(e0.elapsed_time(e1) / 1e3 / args.reps)
    os.environ.pop("CARMA_MULTI_FILTER_STORES", None)
    best = {v: min(ts) for v, ts in times.items()}
    kernels = {}
    for v in variants:
        kernels[v] = {"launch_s": round(best[v], 6), "launch_s_per_round": [round(x, 6) for x in times[v]],
                      "curves_per_s": float("%.4g" % (nc / best[v]))}
        if v != "k4":
            kernels[v]["hbm_bytes_per_s_algorithmic"] = float("%.4g" % (40.0 * total / best[v]))
            kernels[v]["vs_k4"] = round(best[v] / best["k4"], 3)
    kernels["k4"]["hbm_bytes_per_s_algorithmic"] = float("%.4g" % (24.0 * total / best["k4"]))
    checks = {
        "block_equals_scalar_bitwise": bool(all(np.array_equal(a, b) for a, b in zip(outputs["block"], outputs["scalar"]))),
        "loglik_equals_k4_bitwise": bool(np.array_equal(outputs["block"][2], outputs["k4"])),
    }
    del d_mean, d_var
    torch.cuda.empty_cache()

    def wall(fn):
        t0 = time.perf_counter()
        out = fn()   # blocking: returns after its device synchronise
        return time.perf_counter() - t0, out

    m.kalman_filter(kind, p, q, theta[:nc])   # warm-up of the host-array paths
    t_kf, _ = wall(lambda: m.kalman_filter(kind, p, q, theta))
    m.assess_fit_values(kind, p, q, theta, nlags=20)
    t_af, af = wall(lambda: m.assess_fit_values(kind, p, q, theta, nlags=20))
    white = float(np.mean(np.abs(af.acf) < af.bound[:, None]))
    m.close()

    # predict: pcurves curves x nq query times over [-10 %, +110 %] of each curve's span, unsorted
    npc, nq = args.pcurves, args.nq
    mp = C.MultiSeries.simulate(npc, ny, kind, p, q, th, seed=args.seed + 1, **sim)
    span = mp.curve_stats()["tspan"]
    rng = np.random.default_rng(1)
    tq = (rng.uniform(-0.1, 1.1, (npc, nq)) * span[:, None]).reshape(-1)
    qo = np.arange(npc + 1, dtype=np.int64) * nq
    thp = np.tile(th, (npc, 1))
    mp.predict(kind, p, q, thp[:], tq[:], qo)   # warm-up
    t_pr, (qm, qv) = wall(lambda: mp.predict(kind, p, q, thp, tq, qo))

    # what a user does today: one Series per curve, explicit parameters from the theta row
    nsub = min(args.subset, npc)
    der = C._lib.derived_params(kind, p, q, th[None, :])
    s2, roots, ma = der["sigma"][0] ** 2, der["ar_roots"][0], der["ma_coefs"][0]
    curves = [mp.curve(c) for c in range(nsub)]
    t, y, e = curves[0]
    C.Series(t, y, e).filter(s2, roots, ma, measerr_scale=th[1], mu=th[2])   # warm-up
    t0 = time.perf_counter()
    loop_max_dm = 0.0
    for c, (t, y, e) in enumerate(curves):
        s = C.Series(t, y, e)
        s.filter(s2, roots, ma, measerr_scale=th[1], mu=th[2])
        s.close()
    t_loop_f = time.perf_counter() - t0
    t0 = time.perf_counter()
    for c, (t, y, e) in enumerate(curves):
        s = C.Series(t, y, e)
        lm, lv = s.predict(s2, roots, ma, tq[qo[c]:qo[c + 1]], measerr_scale=th[1], mu=th[2])
        s.close()
        loop_max_dm = max(loop_max_dm, float(np.max(np.abs(lm + th[2] - qm[qo[c]:qo[c + 1]]))))
    t_loop_p = time.perf_counter() - t0
    mp.close()

    name, power = card()
    out = {
        "what": "MultiSeries Kalman filter / assess_fit_values / predict, CARMA(3,1) at the true parameters on simulated "
                "curves of ny = %d" % ny,
        "gpu": name, "power_limit": power,
        "filter_kernel": {"curves": nc, "ny": ny, "points": total, "reps_per_window": args.reps, "rounds": args.rounds,
                          "variants": kernels, "checks": checks},
        "kalman_filter_end_to_end": {"curves": nc, "wall_s": round(t_kf, 4), "curves_per_s": float("%.4g" % (nc / t_kf))},
        "assess_fit_values_end_to_end": {"curves": nc, "nlags": 20, "wall_s": round(t_af, 4),
                                         "curves_per_s": float("%.4g" % (nc / t_af)),
                                         "acf_inside_band_fraction": round(white, 4)},
        "predict_end_to_end": {"curves": npc, "queries_per_curve": nq, "wall_s": round(t_pr, 4),
                               "curves_per_s": float("%.4g" % (npc / t_pr)),
                               "queries_per_s": float("%.4g" % (npc * nq / t_pr))},
        "python_loop": {"curves": nsub,
                        "filter_wall_s": round(t_loop_f, 3), "filter_curves_per_s": round(nsub / t_loop_f, 2),
                        "predict_wall_s": round(t_loop_p, 3), "predict_curves_per_s": round(nsub / t_loop_p, 2),
                        "predict_max_abs_diff_vs_survey": loop_max_dm,
                        "what": "Series(curve).filter / .predict(%d times) per curve" % nq},
    }
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
