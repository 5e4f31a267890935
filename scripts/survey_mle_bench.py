"""Survey-scale maximum likelihood on one GPU: CARMA(3,1) fitted to every curve of a simulated survey
(MultiSeries.get_mle: one starting-value launch, one fitting launch), against what a user does without it -- a Python
loop of CarmaModel(curve).get_mle(..., optimizer="device") -- on a subset of the curves.

Reports fits/s, curves/s, total evaluations (sum of nfev) and evaluations/s of the fitting launch, the starting-value
time, and the fraction of curves whose best fit reaches the likelihood of the true parameters.  The card's name and
power limit are read in the same run.

    python scripts/survey_mle_bench.py [--curves 16000] [--ny 500] [--starts 16] [--subset 50] [--out FILE]
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
    ap.add_argument("--curves", type=int, default=16000)
    ap.add_argument("--ny", type=int, default=500)
    ap.add_argument("--starts", type=int, default=16)
    ap.add_argument("--subset", type=int, default=50)
    ap.add_argument("--repeats", type=int, default=2, help="fitting launches (the fastest is reported)")
    ap.add_argument("--seed", type=int, default=17)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import carma_pack_b200 as C
    from carma_pack_b200 import synth
    from carma_pack_b200.carma_pack import _survey_starts
    if C._lib.device_count() < 1:
        raise SystemExit("no CUDA device visible")
    p, q, ns = 3, 1, args.starts
    th = synth.carma31_theta()
    sim = dict(yerr=0.2, dt_min=0.05, dt_max=60.0)

    def sync_time(fn):
        t0 = time.perf_counter()
        out = fn()   # every call below is blocking: it returns after its device synchronise
        return time.perf_counter() - t0, out

    # warm-up of every shape used: the PT and fitting kernels of CARMA(3,1), the single-curve path
    warm = C.MultiSeries.simulate(32, args.ny, C.KIND_CARMA, p, q, th, seed=args.seed + 1, **sim)
    warm.get_mle(p, q, ntrials=ns, seed=1)
    t, y, e = warm.curve(0)
    C.CarmaModel(t, y, e).get_mle(p, q, ntrials=ns, seed=1, optimizer="device")
    warm.close()

    m = C.MultiSeries.simulate(args.curves, args.ny, C.KIND_CARMA, p, q, th, seed=args.seed, **sim)
    stats = m.curve_stats()
    t_starts, (kind, x0, lo, hi, flags) = sync_time(lambda: _survey_starts(m, p, q, ns, 99, 0, None, stats))
    job = [(kind, p, q, x0, lo, hi, flags)]
    fit_times, results = [], []
    for r in range(args.repeats):
        dt, (res,) = sync_time(lambda: m.mle_grid(job))
        fit_times.append(dt)
        results.append(res)
    same = all(np.array_equal(a, b) for res in results[1:] for a, b in zip(results[0], res))
    x, f, nit, nfev = results[0]
    t_fit = min(fit_times)
    nfits = args.curves * ns
    evals = int(nfev.sum())
    f_true = -m.loglik(C.KIND_CARMA, p, q, np.tile(th, (args.curves, 1)), priors=m.default_priors(), flags=C.IGNORE_BOUNDS)
    best = f.min(axis=1)
    recovered = float(np.mean(best <= f_true + 1e-6 * np.abs(best)))

    # what a user does today: one CarmaModel per curve, each with its own starting-value run and fitting launch
    nsub = min(args.subset, args.curves)
    curves = [m.curve(c) for c in range(nsub)]
    t0 = time.perf_counter()
    loop_fun = []
    for c, (t, y, e) in enumerate(curves):
        r = C.CarmaModel(t, y, e).get_mle(p, q, ntrials=ns, seed=99, trial_offset=c * ns, optimizer="device")
        loop_fun.append(r.fun)
    t_loop = time.perf_counter() - t0
    m.close()

    name, power = card()
    out = {
        "what": "MultiSeries.get_mle, CARMA(3,1) fitted from %d starts to each of %d simulated curves of ny = %d"
                % (ns, args.curves, args.ny),
        "gpu": name, "power_limit": power,
        "curves": args.curves, "ny": args.ny, "starts_per_curve": ns, "fits": nfits,
        "starting_values_s": round(t_starts, 4),
        "fit_launch_s": round(t_fit, 4),
        "fits_per_s": round(nfits / t_fit, 1),
        "curves_per_s": round(args.curves / (t_fit + t_starts), 1),
        "evaluations": evals,
        "evaluations_per_s": float("%.4g" % (evals / t_fit)),
        "mean_evaluations_per_fit": round(evals / nfits, 1),
        "max_iterations": int(nit.max()),
        "recovered_fraction": recovered,
        "fit_launch_repeats_s": [round(v, 4) for v in fit_times],
        "repeats_bitwise_equal": bool(same),
        "python_loop": {"curves": nsub, "wall_s": round(t_loop, 3), "curves_per_s": round(nsub / t_loop, 2),
                        "what": "CarmaModel(curve).get_mle(3, 1, ntrials=%d, optimizer='device') per curve" % ns},
        "survey_curves_per_s_vs_loop": round((args.curves / (t_fit + t_starts)) / (nsub / t_loop), 1),
    }
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
