"""Survey-scale posterior summaries on one GPU (carma_psd_quantiles, carma_effective_samples), against what a user does
without them -- a Python loop of CarmaSample.psd_credible_band + effective_samples -- on a subset of the curves.

  * the band: --curves CARMA(3,1) traces of --samples rows around the survey truth, --nfreq log-spaced frequencies,
    three percentiles (16, 84, 50).  Device time of carma_psd_quantiles_dev (CUDA events, every kernel of the call) and
    the end-to-end time of carma_psd_quantiles from host arrays (copies, chunks, synchronise); best of --reps;
  * the global-memory path at --long-samples samples per curve on --long-curves curves (device time);
  * the ESS kernel on the same trace (all seven columns), device time; the rows of that trace are independent, so the
    kernel stops at lag 1 and this is its lower bound -- it is also timed on an AR(1) trace (phi = 0.9, tau ~ 19) of the
    same shape, where it runs tens of lags;
  * the Python loop over --subset curves, given as curves/s (the CarmaSample construction, one derived-parameter
    launch per curve, is timed apart).
The working set of every timed call is larger than the 126 MB L2.  The card's name and power limit are read in the same run.

    python scripts/survey_posterior_bench.py [--curves 10000] [--samples 1000] [--nfreq 200] [--out FILE]
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


def traces(nc, ns, seed):
    from carma_pack_b200 import synth
    ar, ma, s2 = synth.carma31_truth()
    tail = np.concatenate([synth.roots_to_logquad(ar), [np.log(ma[1])]])
    rng = np.random.default_rng(seed)
    th = np.empty((nc, ns, 7))
    th[:, :, 0] = np.sqrt(synth.carma_variance(s2, ar, ma).real) * rng.uniform(0.8, 1.2, (nc, ns))
    th[:, :, 1] = rng.uniform(0.9, 1.1, (nc, ns))
    th[:, :, 2] = rng.normal(0.0, 0.1, (nc, ns))
    th[:, :, 3:] = tail + rng.normal(0.0, 0.05, (nc, ns, 4))
    return th


def device_time(fn, reps):
    import torch
    fn()
    torch.cuda.synchronize()
    best = np.inf
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        best = min(best, a.elapsed_time(b) * 1e-3)
    return best


def band_dev(C, th_d, fr_d, pct_d, out_d, nc, ns, nf):
    def run():
        C._lib.check(C._lib.lib.carma_psd_quantiles_dev(C.KIND_CARMA, 3, 1, None, nc, ns, th_d.data_ptr(), fr_d.data_ptr(), 1,
                                                          nf, pct_d.data_ptr(), 3, out_d.data_ptr(), None, None),
                     "carma_psd_quantiles_dev")
    return run


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--curves", type=int, default=10000)
    ap.add_argument("--samples", type=int, default=1000)
    ap.add_argument("--nfreq", type=int, default=200)
    ap.add_argument("--long-curves", type=int, default=100)
    ap.add_argument("--long-samples", type=int, default=64000)
    ap.add_argument("--subset", type=int, default=100)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import carma_pack_b200 as C
    name, power = card()
    nc, ns, nf = a.curves, a.samples, a.nfreq
    pct = np.array([16.0, 84.0, 50.0])
    th = traces(nc, ns, seed=1)
    fr = np.logspace(-3.5, 0.5, nf)
    dev = torch.device("cuda:0")
    th_d = torch.from_numpy(th).to(dev)
    fr_d, pct_d = torch.from_numpy(fr).to(dev), torch.from_numpy(pct).to(dev)
    out_d = torch.empty((nc, 3, nf), dtype=torch.float64, device=dev)
    res = {"card": name, "power_limit": power, "curves": nc, "samples": ns, "nfreq": nf, "percentiles": pct.tolist()}

    t_band = device_time(band_dev(C, th_d, fr_d, pct_d, out_d, nc, ns, nf), a.reps)
    res["band_device_s"] = round(t_band, 5)
    evals = nc * ns * nf
    res["band_psd_evals_per_s"] = evals / t_band
    best = np.inf
    for _ in range(a.reps):
        t0 = time.perf_counter()
        host = C._lib.psd_quantiles(C.KIND_CARMA, 3, 1, th, fr, pct)
        best = min(best, time.perf_counter() - t0)
    res["band_end_to_end_s"] = round(best, 4)
    assert np.array_equal(host, out_d.cpu().numpy())

    # selection paths at the benchmark size: the global path (radix select over a scratch column) for comparison
    os.environ["CARMA_PSD_GLOBAL_SELECT"] = "1"
    res["band_device_s_global_path"] = round(device_time(band_dev(C, th_d, fr_d, pct_d, out_d, nc, ns, nf), a.reps), 5)
    assert np.array_equal(host, out_d.cpu().numpy())
    del os.environ["CARMA_PSD_GLOBAL_SELECT"]

    # ESS of every column of the same trace
    ess_d = torch.empty((nc, 7), dtype=torch.float64, device=dev)

    def ess_run():
        C._lib.check(C._lib.lib.carma_effective_samples_dev(nc, ns, 7, th_d.data_ptr(), ess_d.data_ptr(), None),
                     "carma_effective_samples_dev")
    res["ess_device_s_iid_trace"] = round(device_time(ess_run, a.reps), 5)
    ess_host = ess_d.cpu().numpy()
    ar1 = np.empty((ns, nc, 7))
    rng = np.random.default_rng(3)
    ar1[0] = rng.standard_normal((nc, 7))
    for i in range(1, ns):
        ar1[i] = 0.9 * ar1[i - 1] + rng.standard_normal((nc, 7))
    ar1 = np.ascontiguousarray(ar1.transpose(1, 0, 2))
    th_d.copy_(torch.from_numpy(ar1))
    res["ess_device_s_ar1_phi0.9"] = round(device_time(ess_run, a.reps), 5)
    ess_ar1 = ess_d.cpu().numpy()
    res["ess_ar1_median"] = float(np.median(ess_ar1))
    assert np.allclose(ess_ar1[0], [MS_ess(C, ar1[0][:, j]) for j in range(7)], rtol=1e-10, atol=0)
    del ar1
    del th_d, out_d, ess_d
    torch.cuda.empty_cache()

    # the Python loop over a subset
    k = min(a.subset, nc)
    t0 = time.perf_counter()
    samples = [C.CarmaSample(np.arange(5.0), np.zeros(5), np.ones(5), trace=th[c], logpost=np.zeros(ns), p=3, q=1)
               for c in range(k)]
    t_build = time.perf_counter() - t0
    t0 = time.perf_counter()
    for c, cs in enumerate(samples):
        lo, hi, mid, _ = cs.psd_credible_band(percentile=68.0, nsamples=None, freq=fr)
        e = np.array([MS_ess(C, th[c][:, j]) for j in range(7)])
    t_loop = time.perf_counter() - t0
    assert np.allclose(np.stack([lo, hi, mid]), host[k - 1], rtol=1e-8, atol=0)
    assert np.allclose(e, ess_host[k - 1], rtol=1e-10, atol=0)
    res["python_loop_curves"] = k
    res["python_loop_band_ess_curves_per_s"] = k / t_loop
    res["python_loop_carmasample_build_s_per_curve"] = t_build / k
    res["survey_band_curves_per_s_end_to_end"] = nc / res["band_end_to_end_s"]

    # global path at long columns
    lc, ls = a.long_curves, a.long_samples
    thl = traces(lc, ls, seed=2)
    thl_d = torch.from_numpy(thl).to(dev)
    outl_d = torch.empty((lc, 3, nf), dtype=torch.float64, device=dev)
    del thl
    res["long_curves"], res["long_samples"] = lc, ls
    res["long_band_device_s"] = round(device_time(band_dev(C, thl_d, fr_d, pct_d, outl_d, lc, ls, nf), max(2, a.reps // 2)), 5)
    res["long_band_psd_evals_per_s"] = lc * ls * nf / res["long_band_device_s"]
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


def MS_ess(C, col):
    ms = C.MCMCSample()
    ms._samples["x"] = col
    return ms.effective_samples("x")[0]


if __name__ == "__main__":
    main()
