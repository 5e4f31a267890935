"""Survey-scale Laplace importance sampling on one GPU (MultiSeries.laplace_sample / carma_multi_laplace) against the
way to get a posterior and its PSD band without it: run_mcmc.

  * workload: --curves and --curves-large simulated CARMA(3,1) curves of --ny points, fitted with get_mle (outside the
    timed window);
  * timed path, end to end (host arrays in and out, blocking calls), best of --reps after a warm-up: hessian +
    laplace_sample (--draws draws per curve) + psd_credible_band at the fits; the comparison on the --curves curves:
    run_mcmc(--draws) + psd_credible_band;
  * device time per kernel from torch.profiler (CUDA activities) in a separate call, and the evaluation kernel's rate in
    evaluations/s next to multi_hessian_eval_kernel's in the same call.  The rate counts the draws of the curves that
    are not BAD_COV (the kernel returns at once for the others), and the share of those draws that the prior rejects
    (they skip the filter) is reported next to it; the hessian rate counts every stencil point;
  * the fraction of curves with k-hat <= 0.7, and on those the agreement of the 68 % PSD band with MCMC's (|log PSD
    difference| over the MCMC band's log width, median and 90th percentile over curves and frequencies).
The card's name and power limit are read in the same run.

    python scripts/survey_laplace_bench.py [--curves 10000] [--curves-large 100000] [--ny 1000] [--draws 1000] [--out F]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

KERNELS = ("multi_hessian_eval_kernel", "multi_hessian_assemble_kernel", "multi_laplace_factor_kernel",
           "multi_laplace_eval_kernel", "multi_laplace_summary_kernel", "psd_", "pt_kernel", "multi_pt")


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
                break
    return {k: {"device_s": round(out[k], 6), "launches": launches[k]} for k in KERNELS if launches[k]}


def timed(call, reps):
    first = call()   # warm-up: module load, scratch growth
    walls = []
    for _ in range(reps):
        t0 = time.perf_counter()
        call()
        walls.append(time.perf_counter() - t0)
    return first, {"wall_s": round(min(walls), 4), "wall_s_per_rep": [round(w, 4) for w in walls]}


def band_agreement(a, b, keep):
    """|log PSD difference| of band a against band b over b's log width, over the kept curves and every frequency."""
    width = np.log(b[1][keep]) - np.log(b[0][keep])
    err = np.concatenate([(np.abs(np.log(x[keep]) - np.log(y[keep])) / width).ravel() for x, y in zip(a[:3], b[:3])])
    err = err[np.isfinite(err)]
    return {"median": float("%.3g" % np.median(err)), "p90": float("%.3g" % np.quantile(err, 0.9))}


def case(C, p, q, th, nc, ny, draws, reps, seed, ntrials, mcmc):
    kind = C.KIND_CARMA
    m = C.MultiSeries.simulate(nc, ny, kind, p, q, th, yerr=0.2, dt_min=0.05, dt_max=60.0, seed=seed)
    fit = m.get_mle(p, q, ntrials=ntrials, seed=seed + 1)

    def laplace_path():
        ls = m.laplace_sample(p, q, fit.x, ndraws=draws, seed=seed + 2)
        return ls, ls.psd_credible_band(68.0)

    (ls, band), rl = timed(laplace_path, reps)
    rl["kernels"] = kernel_split(laplace_path)
    ks = rl["kernels"]
    d = th.size
    ev, hev = ks["multi_laplace_eval_kernel"]["device_s"], ks["multi_hessian_eval_kernel"]["device_s"]
    good = (ls.status == C.LAPLACE_OK) & (ls.khat <= 0.7)
    # the evaluation kernel returns at once for every draw of a BAD_COV curve, so only the other curves' draws are
    # evaluations; of those, the draws the prior rejects (-inf) skip the filter as well
    evaluated = ls.status != C.LAPLACE_BAD_COV
    n_eval = int(evaluated.sum()) * draws
    rejected = int(np.sum(ls.laplace.logpost[evaluated] == -np.inf))
    hstat = m.hessian(kind, p, q, fit.x).status
    res = {
        "model": "CARMA(%d,%d)" % (p, q), "curves": nc, "ny": ny, "d": d, "draws": draws, "fit_ntrials": ntrials,
        "laplace": rl,
        "laplace_eval_kernel_evaluated_draws": n_eval,
        "laplace_eval_kernel_evaluations_per_s": float("%.3g" % (n_eval / ev)),
        "laplace_prior_rejected_share_of_evaluated_draws": round(rejected / max(n_eval, 1), 4),
        "hessian_eval_kernel_evaluations_per_s": float("%.3g" % (nc * (d * d + d + 1) / hev)),
        "eval_rate_vs_hessian_eval": round((n_eval / ev) / (nc * (d * d + d + 1) / hev), 3),
        "hessian_status_counts": {str(s): int(n) for s, n in zip(*np.unique(hstat, return_counts=True))},
        "status_counts": {str(s): int(n) for s, n in zip(*np.unique(ls.status, return_counts=True))},
        "fraction_khat_le_0p7": round(float(good.mean()), 4),
        "khat_quantiles_10_50_90": [float("%.3g" % v) for v in np.nanquantile(ls.khat[ls.status == 0], [0.1, 0.5, 0.9])],
    }
    if mcmc:
        def mcmc_path():
            s = m.run_mcmc(p, q, draws, seed=seed + 3)
            return s, s.psd_credible_band(68.0)

        (ms, mband), rm = timed(mcmc_path, max(1, reps - 1))
        res["mcmc"] = rm
        res["speedup_end_to_end_vs_mcmc"] = round(rm["wall_s"] / rl["wall_s"], 2)
        res["band_agreement_with_mcmc_khat_le_0p7"] = band_agreement(band, mband, good)
    m.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--curves", type=int, default=10000)
    ap.add_argument("--curves-large", type=int, default=100000)
    ap.add_argument("--ny", type=int, default=1000)
    ap.add_argument("--draws", type=int, default=1000)
    ap.add_argument("--ntrials", type=int, default=8)
    ap.add_argument("--reps", type=int, default=2)
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
    res = []
    for nc, mcmc in ((args.curves, True), (args.curves_large, False)):
        res.append(case(C, 3, 1, th31, nc, args.ny, args.draws, args.reps, args.seed, args.ntrials, mcmc))
        print(json.dumps(res[-1]), flush=True)
    out = {
        "what": "hessian + laplace_sample + psd_credible_band at the get_mle fits vs run_mcmc + psd_credible_band, "
                "simulated CARMA(3,1) curves",
        "gpu": name, "power_limit": power, "cases": res,
    }
    print(json.dumps(out))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
