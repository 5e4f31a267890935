#!/usr/bin/env python
"""bench.py -- headline benchmark of the CARMA(p,q) Kalman log-likelihood hot path on B200.

Metric (BASELINE.json): CARMA(5,3) ny=270 log-likelihood evals/s.  One "step" = one pass of the hot
path over one batch of synthetic input = 65,536 LogDensity evaluations per GPU on one ny=270 light
curve (BASELINE config 2).  With N GPUs every rank evaluates its own 65,536-row batch (weak
scaling, no data-path collective).  The PT-MCMC secondary metric (ensemble-iterations/s, BASELINE
config 3) is measured in the same run and reported under "pt_mcmc".

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

P, Q, NY, NTHETA = 5, 3, 270, 65536
METRIC = "CARMA(5,3) ny=270 loglik evals/s"
UNIT = "evals/s"


def f_step(p):
    """Algorithmic FP64 flops per Kalman step (SURVEY 8d): 20p^2 + 36p + 7, transcendentals excluded."""
    return 20 * p * p + 36 * p + 7


def f_eval(p, ny):
    f_reset = (2.0 / 3.0) * 8 * p ** 3 + 14 * p * p + 8 * p * p
    return (ny - 1) * f_step(p) + f_reset


def load_synth():
    """carma_pack_b200/synth.py (numpy only) loaded BY PATH: the reference arm must not import the product
    package (importing it loads libcarma_b200.so)."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("_bench_synth", os.path.join(ROOT, "carma_pack_b200", "synth.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def make_inputs(seed_offset=0):
    synth = load_synth()
    t, y, e = synth.readme_series(NY, 270)
    th = synth.theta_batch(NTHETA, t, y, p=P, q=Q, seed=1000 + seed_offset)
    return t, y, e, th


def workload_config():
    """The `config` object: identical in both arms (the driver compares them)."""
    return {"workload": "batched log-likelihood: 65,536 CARMA(5,3) parameter vectors on one ny=270 series per GPU "
                        "(BASELINE config 2)", "p": P, "q": Q, "ny": NY, "thetas_per_step": NTHETA}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.sm_max = None
        self._halt = threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                if len(f) >= 6:
                    self.samples.append(float(f[0]))
                    self.sm_max = float(f[1])
                    for nm, v in zip(names, f[2:6]):
                        if v.lower().startswith("active"):
                            self.reasons.add(nm)
            except Exception:
                pass
            self._halt.wait(0.1)

    def stop(self):
        self._halt.set()
        self.join(timeout=5)
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None,
                "sm_max_mhz": self.sm_max, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def _oracle_worker(args):
    from oracle import oracle as O
    t, y, e, th, lean = args
    pr = O.default_prior(t, y)
    return O.logdensity(O.KIND_CARMA, P, Q, t, y, e, th, prior=pr, fast=True, lean=lean)


def cpu_oracle_rate(t, y, e, th, cores, lean=False):
    """evals/s of the CPU oracle (oracle/carma_oracle.cpp, -O3 x86-64-v3) on `cores` processes.
    lean: the fixed-size heap-free variant instead of the dense as-written one (BASELINE.md section 3)."""
    from oracle import oracle as O
    O.build()
    if cores == 1:
        t0 = time.perf_counter()
        _oracle_worker((t, y, e, th, lean))
        return th.shape[0] / (time.perf_counter() - t0)
    import multiprocessing as mp
    chunks = np.array_split(th, cores)
    with mp.get_context("fork").Pool(cores) as pool:
        pool.map(_oracle_worker, [(t, y, e, c[:64], lean) for c in chunks])  # warm the pool
        t0 = time.perf_counter()
        pool.map(_oracle_worker, [(t, y, e, c, lean) for c in chunks])
        dt = time.perf_counter() - t0
    return th.shape[0] / dt


def run_reference(args, rank, world):
    """Reference arm: the reference's CPU algorithm for this path (oracle port; the reference itself
    needs Armadillo+Boost and cannot be built here) on all host cores, same config/metric/unit."""
    if rank != 0:
        return
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    t, y, e, th = make_inputs()
    sample = th[:16384] if cores < 16 else th
    if args.warmup > 0:
        cpu_oracle_rate(t, y, e, sample[:2048], cores)
    t0 = time.perf_counter()
    rates = [cpu_oracle_rate(t, y, e, sample, cores) for _ in range(args.steps)]
    wall = time.perf_counter() - t0
    value = float(np.mean(rates))
    lean = float(cpu_oracle_rate(t, y, e, sample, cores, lean=True))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * wall / max(args.steps, 1), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "variant": "dense as-written (per-call vector copies, full p x p complex products)",
                         "lean_variant_value": lean,
                         "lean_variant": "same arithmetic, fixed-size arrays, no heap in the time loop (bitwise equal results)",
                         "sample": "%d of the 65,536 theta rows per step, split over %d processes" % (sample.shape[0], cores)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def _reduce_secondary(dist, torch, ms, err):
    """max-over-ranks time of a secondary measurement; every rank calls this (also after a local failure), so a
    rank that failed cannot leave the others waiting in a collective."""
    failed = 0.0 if err is None else 1.0
    if dist:
        tt = torch.tensor([ms if err is None else -1.0, failed], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms, failed = float(tt[0].item()), float(tt[1].item())
    return ms, failed > 0


def run_ours(args, rank, world, local_rank):
    import torch
    import carma_pack_b200 as C
    import ctypes

    if not torch.cuda.is_available() or C._lib.device_count() < 1:
        raise RuntimeError("bench.py: no CUDA device; the product path has no CPU fallback")
    dev = local_rank
    torch.cuda.set_device(dev)
    dist = None
    if world > 1:
        import torch.distributed as dist
        # NCCL announces its version on stdout when the communicator is created; keep stdout for the
        # single JSON line by pointing fd 1 at stderr while the communicator comes up.
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", dev))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)

    t, y, e, th = make_inputs(seed_offset=rank)
    series = C.Series(t, y, e, device=dev)
    prior = series.default_prior()
    d = th.shape[1]
    d_theta = torch.from_numpy(th).to("cuda", non_blocking=False)
    d_out = torch.empty(NTHETA, dtype=torch.float64, device="cuda")
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device="cuda")  # 256 MB > 126 MB L2
    stream = torch.cuda.current_stream().cuda_stream

    def step():
        series.loglik_dev(C.KIND_CARMA, P, Q, d_theta.data_ptr(), d_out.data_ptr(), NTHETA, prior, 0, stream)

    W, K = max(args.warmup, 3), args.steps
    for _ in range(W):
        step()
    torch.cuda.synchronize()
    fp64_peak = C._lib.fp64_peak_tflops(dev)  # measured DFMA saturation on this GPU, before the timed region

    sampler = ClockSampler(dev) if rank == 0 else None
    if sampler:
        sampler.start()
    if dist:
        dist.barrier()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    for k in range(K):
        flush.zero_()  # L2 flush between timed iterations, outside the per-step event pair
        ev[k][0].record()
        step()
        ev[k][1].record()
    torch.cuda.synchronize()
    if dist:
        dist.barrier()
    step_ms = [a.elapsed_time(b) for a, b in ev]
    # what the last timed step handed its caller, copied out after its timing has been read
    last_out = d_out.cpu().numpy() if args.dump_outputs and rank == 0 else None
    total_ms = float(sum(step_ms))
    if dist:
        tt = torch.tensor([total_ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        total_ms = float(tt.item())
    # ---- the same measurement restricted to the in-prior rows (SURVEY 8d: out-of-prior draws are kept in the
    # headline batch because the sampler meets them too, but they leave the kernel after the prologue)
    fin_idx = torch.nonzero(torch.isfinite(d_out)).flatten()
    n_fin = int(fin_idx.numel())
    d_theta_fin = d_theta.index_select(0, fin_idx).contiguous()
    d_out_fin = torch.empty(n_fin, dtype=torch.float64, device="cuda")
    series.loglik_dev(C.KIND_CARMA, P, Q, d_theta_fin.data_ptr(), d_out_fin.data_ptr(), n_fin, prior, 0, stream)
    torch.cuda.synchronize()
    fin_ms = 0.0
    ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(K):
        flush.zero_()
        ea.record()
        series.loglik_dev(C.KIND_CARMA, P, Q, d_theta_fin.data_ptr(), d_out_fin.data_ptr(), n_fin, prior, 0, stream)
        eb.record()
        torch.cuda.synchronize()
        fin_ms += ea.elapsed_time(eb)
    fin_rate = n_fin * K / (fin_ms * 1e-3)
    if dist:
        tt = torch.tensor([fin_rate], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.SUM)
        fin_rate = float(tt.item())
    in_prior = {"rows_rank0": n_fin, "ms_per_step_rank0": fin_ms / K, "value": fin_rate, "unit": UNIT,
                "all_finite": bool(torch.isfinite(d_out_fin).all().item())}

    # the clock sampler keeps running through the e2e / PT-MCMC / survey / scan measurements below so that
    # several nvidia-smi samples fall inside timed regions (the K-step region alone lasts ~10 ms)

    # ---- end-to-end through the host-buffer C-ABI calls (pinned host memory; every step does its own
    # H2D of the 65,536 x 11 theta block and D2H of the 65,536 results inside the timed region).
    # Two forms: the blocking call, and the two-slot pipelined call (copies of step k+1 overlap the kernel
    # of step k) which is what a host-driven caller evaluating batch after batch would use.
    NSLOT = 4   # CARMA_N_SLOTS: steps in flight; with two, the H2D of a step could not start before the step two back had been waited for
    h_theta = [torch.from_numpy(th.copy()).pin_memory() for _ in range(NSLOT)]
    h_outs = [torch.empty(NTHETA, dtype=torch.float64).pin_memory() for _ in range(NSLOT)]
    h_out = h_outs[0]
    lib = C._lib.lib

    def e2e_step():
        C._lib.check(lib.carma_loglik_batch(series.handle, C.KIND_CARMA, P, Q, ctypes.byref(prior), NTHETA,
                                            h_theta[0].data_ptr(), h_out.data_ptr(), 0), "carma_loglik_batch")

    E2E_REPEATS = 5   # the K-step region lasts a few ms: repeat it and report the median (max over ranks per repeat)
    for _ in range(3):
        e2e_step()
    block_s = []
    for _ in range(E2E_REPEATS):
        if dist:
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(K):
            e2e_step()  # synchronous: returns after the D2H copy completed
        block_s.append(time.perf_counter() - t0)

    def e2e_pipelined(nsteps):
        for k in range(nsteps):
            slot = k % NSLOT
            if k >= NSLOT:
                series.loglik_wait(slot)      # results of step k-NSLOT are in h_outs[slot]; its buffers are free again
            series.loglik_async(C.KIND_CARMA, P, Q, h_theta[slot].data_ptr(), h_outs[slot].data_ptr(), NTHETA, prior, slot)
        for slot in range(NSLOT):
            series.loglik_wait(slot)

    e2e_pipelined(2 * NSLOT)
    # the box's host-to-device rate for one step's theta block (pinned), to read the e2e figure against
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    h2d_ms = []
    d_scratch = torch.empty_like(d_theta)
    for _ in range(5):
        ev0.record()
        d_scratch.copy_(h_theta[0].view_as(d_theta), non_blocking=True)
        ev1.record()
        ev1.synchronize()
        h2d_ms.append(ev0.elapsed_time(ev1))
    h2d_gbs = NTHETA * d * 8 / (float(np.median(h2d_ms)) * 1e-3) / 1e9
    del d_scratch
    pipe_s = []
    for _ in range(E2E_REPEATS):
        if dist:
            dist.barrier()
        t0 = time.perf_counter()
        e2e_pipelined(K)
        pipe_s.append(time.perf_counter() - t0)
    if dist:
        tt = torch.tensor(pipe_s + block_s, dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        pipe_s, block_s = [float(x) for x in tt[:E2E_REPEATS]], [float(x) for x in tt[E2E_REPEATS:]]
    e2e_s, e2e_block_s = float(np.median(pipe_s)), float(np.median(block_s))
    checksum = float(np.nansum(np.where(np.isfinite(h_out.numpy()), h_out.numpy(), 0.0)))
    same = bool(np.array_equal(h_out.numpy(), d_out.cpu().numpy(), equal_nan=True))

    # ---- PT-MCMC secondary metric (BASELINE config 3 shape: 10 temperatures, ny=1000, on-device adapt/exchange)
    # (secondary measurements are guarded: a failure is reported in their own block, never in place of the line)
    pt = None
    if not args.no_pt:
        from carma_pack_b200 import synth
        n_ens = args.pt_ensembles
        pt_ms, pt_err, iters, pt_finite, sp = 0.0, None, 0, False, None
        try:
            tp, yp, ep = synth.readme_series(1000, 1000)
            sp = C.Series(tp, yp, ep, device=dev)
            ppr = sp.default_prior()
            o = C.PTOpts()
            lib.carma_pt_default_opts(ctypes.byref(o))
            o.nsamples, o.burnin, o.thin, o.ntemps = args.pt_iters // 2, args.pt_iters - args.pt_iters // 2, 1, 10
            o.seed, o.ensemble_offset = 4096, rank * n_ens
            iters = o.burnin + o.nsamples
            ds = torch.empty(n_ens * o.nsamples * d, dtype=torch.float64, device="cuda")
            dl = torch.empty(n_ens * o.nsamples, dtype=torch.float64, device="cuda")
            o_w = C.PTOpts.from_buffer_copy(o)
            o_w.nsamples, o_w.burnin = 1, 1
            sp.pt_run_dev(C.KIND_CARMA, P, Q, o_w, n_ens, ds.data_ptr(), dl.data_ptr(), ppr, stream=stream)  # warm-up
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            sp.pt_run_dev(C.KIND_CARMA, P, Q, o, n_ens, ds.data_ptr(), dl.data_ptr(), ppr, stream=stream)
            b.record()
            torch.cuda.synchronize()
            pt_ms = a.elapsed_time(b)
            pt_finite = bool(torch.isfinite(dl).all().item())
            del ds, dl
        except Exception as ex:  # noqa: BLE001
            pt_err = "%s: %s" % (type(ex).__name__, ex)
        finally:
            if sp is not None:
                sp.close()
        pt_ms, pt_failed = _reduce_secondary(dist, torch, pt_ms, pt_err)
        if pt_failed:
            pt = {"error": pt_err or "failed on another rank"}
        else:
            # the launch also draws starting values: (iters + ~1 start eval) evals per chain
            pt = {"metric": "PT-MCMC ensemble-iterations/s, CARMA(5,3), ny=1000, 10 temperatures, order=reference(pipelined)",
                  "value": world * n_ens * iters / (pt_ms * 1e-3), "unit": "ensemble-iters/s",
                  "implied_evals_per_s": world * n_ens * iters * 10 / (pt_ms * 1e-3),
                  "ensembles_per_gpu": n_ens, "iterations": iters, "ms": pt_ms, "kernel_launches": 1,
                  "includes": "starting-value draws (>= 1 log-density per chain) and the ntemps-1 fill/drain ticks of the "
                              "pipelined reference step order, all inside the one timed launch",
                  "tflops_algorithmic": world * n_ens * iters * 10 * f_eval(P, 1000) / (pt_ms * 1e-3) / 1e12,
                  "finite_logposts": pt_finite}

    # ---- survey-scale secondary metric (BASELINE config 5): one CARMA(3,1) theta per light curve, ny = 1000
    survey = None
    if not args.no_survey:
        from carma_pack_b200 import synth
        # BASELINE config 5 is a FIXED survey (10^6 curves) spread over the GPUs: strong scaling
        ncv, nyc = max(1, args.survey_curves // world), 1000
        sv_ms, sv_err, t_gen, sv_finite, ms_ = 0.0, None, 0.0, 0.0, None
        try:
            rng = np.random.default_rng(5000 + rank)
            # the light curves are drawn from the CARMA(3,1) truth ON the device (carma_multi_series_simulate):
            # 24 bytes per point never cross PCIe, which is what lets one GPU hold the 10^6-curve survey
            th_true = synth.carma31_theta(sigmay=1.0, mu=0.0)
            t_gen = time.perf_counter()
            ms_ = C.MultiSeries.simulate(ncv, nyc, C.KIND_CARMA, 3, 1, th_true, yerr=0.3, dt_min=0.1, dt_max=1e3,
                                         seed=5000, curve_offset=rank * ncv, device=dev)
            t_gen = time.perf_counter() - t_gen
            th31 = np.tile(th_true, (ncv, 1))
            th31[:, 3:] += 0.05 * rng.standard_normal((ncv, 4))
            d_pr = torch.from_numpy(ms_.default_priors().view(np.float64).reshape(ncv, 6)).cuda()
            d_th = torch.from_numpy(th31).cuda()
            d_o = torch.empty(ncv, dtype=torch.float64, device="cuda")
            for _ in range(2):
                ms_.loglik_dev(C.KIND_CARMA, 3, 1, d_pr.data_ptr(), d_th.data_ptr(), d_o.data_ptr(), 0, stream)
            torch.cuda.synchronize()
            reps = 5
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            tot = 0.0
            for _ in range(reps):
                flush.zero_()
                a.record()
                ms_.loglik_dev(C.KIND_CARMA, 3, 1, d_pr.data_ptr(), d_th.data_ptr(), d_o.data_ptr(), 0, stream)
                b.record()
                torch.cuda.synchronize()
                tot += a.elapsed_time(b)
            sv_ms = tot / reps
            sv_finite = float(torch.isfinite(d_o).float().mean().item())
            del d_pr, d_th, d_o
        except Exception as ex:  # noqa: BLE001
            sv_err = "%s: %s" % (type(ex).__name__, ex)
        finally:
            if ms_ is not None:
                ms_.close()
        sv_ms, sv_failed = _reduce_secondary(dist, torch, sv_ms, sv_err)
        if sv_failed:
            survey = {"error": sv_err or "failed on another rank"}
        else:
            survey = {"metric": "multi light-curve LogDensity, CARMA(3,1), ny=1000, one theta per curve",
                      "value": world * ncv / (sv_ms * 1e-3), "unit": "curves/s", "curves_per_gpu": ncv, "ms": sv_ms,
                      "curves_total": world * ncv, "scaling": "strong (the survey is split over the ranks, max-over-ranks time)",
                      "hbm_gbs_algorithmic": ncv * nyc * 24 / (sv_ms * 1e-3) / 1e9,
                      "tflops_algorithmic": ncv * f_eval(3, nyc) / (sv_ms * 1e-3) / 1e12,
                      "finite": sv_finite,
                      "generate_s": t_gen,
                      "data": "synthetic, generated in HBM: Cauchy-gap times (generate_test_data.py:17), CARMA(3,1) draws + N(0,0.3^2) noise"}

    # ---- single very long series through the associative-scan kernel (BASELINE config 5, ny = 10^6)
    scan = None
    if not args.no_scan and rank == 0:
        sl = None
        try:
            from carma_pack_b200 import synth
            nl = args.scan_ny
            rng = np.random.default_rng(77)
            tl = np.cumsum(rng.uniform(0.5, 1.5, nl))
            sl = C.Series(tl, rng.standard_normal(nl), np.full(nl, 0.3), device=dev)
            ar31, _, _ = synth.carma31_truth()
            th1 = torch.tensor([[1.0, 1.0, 0.0] + list(synth.roots_to_logquad(ar31)) + [np.log(1.0 / 3.0)]], dtype=torch.float64).cuda()
            o1 = torch.empty(1, dtype=torch.float64, device="cuda")
            o2 = torch.empty(1, dtype=torch.float64, device="cuda")
            prl = sl.default_prior()
            sl.loglik_scan_dev(C.KIND_CARMA, 3, 1, th1.data_ptr(), o1.data_ptr(), 1, prl, C.IGNORE_BOUNDS, 0, stream)
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(5):
                sl.loglik_scan_dev(C.KIND_CARMA, 3, 1, th1.data_ptr(), o1.data_ptr(), 1, prl, C.IGNORE_BOUNDS, 0, stream)
            b.record()
            torch.cuda.synchronize()
            scan_ms = a.elapsed_time(b) / 5
            a.record()
            sl.loglik_dev(C.KIND_CARMA, 3, 1, th1.data_ptr(), o2.data_ptr(), 1, prl, C.IGNORE_BOUNDS, stream)
            b.record()
            torch.cuda.synchronize()
            seq_ms = a.elapsed_time(b)
            scan = {"metric": "one CARMA(3,1) LogDensity on a single ny=%d series, associative-scan kernels (5 launches)" % nl,
                    "ms": scan_ms, "points_per_s": nl / (scan_ms * 1e-3), "sequential_one_thread_ms": seq_ms,
                    "rel_diff_vs_sequential": abs(float(o1.item()) - float(o2.item())) / abs(float(o2.item()))}
        except Exception as ex:  # noqa: BLE001
            scan = {"error": "%s: %s" % (type(ex).__name__, ex)}
        finally:
            if sl is not None:
                sl.close()

    # ---- choose_order secondary (BASELINE config 4): pmax = 7 (28 models) x 100 random starts on an ny = 500 series;
    # the (model, start) grid is sharded over the ranks by cost and only per-model summaries are all-gathered
    order = None
    if not args.no_order:
        o_err, o_wall, o_sel, o_best = None, 0.0, None, None
        try:
            from carma_pack_b200 import synth
            t5, y5, e5 = synth.readme_series(500, 500)
            model = C.CarmaModel(t5, y5, e5, device=dev)
            model.choose_order(7, ntrials=2, seed=1, verbose=False, dist=dist)   # warm-up: every order's kernels loaded, series, streams
            if dist:
                dist.barrier()
            t0 = time.perf_counter()
            best, pq, aicc = model.choose_order(7, ntrials=args.order_trials, seed=500, verbose=False, dist=dist)
            o_wall = time.perf_counter() - t0
            o_sel, o_best = [int(model.p), int(model.q)], float(np.min(aicc))
            aicc_table = [float(a) for a in aicc]
        except Exception as ex:  # noqa: BLE001
            o_err = "%s: %s" % (type(ex).__name__, ex)
        o_wall, o_failed = _reduce_secondary(dist, torch, o_wall * 1e3, o_err)
        if o_failed:
            order = {"error": o_err or "failed on another rank"}
        else:
            order = {"metric": "choose_order(pmax=7) wall time, 28 (p,q) models x %d starts, ny=500" % args.order_trials,
                     "wall_s": o_wall * 1e-3, "selected_pq": o_sel, "best_aicc": o_best, "aicc": aicc_table,
                     "scaling": "strong (one grid, sharded over %d rank(s) by cost)" % world}

    clocks = sampler.stop() if sampler else None

    # ---- NCCL: gather per-rank summaries only (no data-path collective)
    summary = [float(torch.nan_to_num(d_out, neginf=-1e300).max().item()), float(torch.isfinite(d_out).sum().item())]
    if dist:
        g = [torch.zeros(2, dtype=torch.float64, device="cuda") for _ in range(world)]
        dist.all_gather(g, torch.tensor(summary, dtype=torch.float64, device="cuda"))
        summary = [max(float(x[0]) for x in g), sum(float(x[1]) for x in g)]

    if rank == 0:
        evals = world * NTHETA * K
        value = evals / (total_ms * 1e-3)
        kern_ms = float(np.mean(step_ms))
        fe = f_eval(P, NY)
        achieved_tf = NTHETA * fe / (kern_ms * 1e-3) / 1e12
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        alg_bytes = NTHETA * (8 * d + 8) + 24 * NY
        # CPU baseline beside it: oracle port, one core, the same 65,536-row batch (about 5-8 s)
        cpu = None
        if not args.no_cpu:
            rate1 = float(np.mean([cpu_oracle_rate(t, y, e, th, 1) for _ in range(2)]))
            lean1 = float(cpu_oracle_rate(t, y, e, th, 1, lean=True))
            cpu = {"value": rate1, "unit": UNIT, "cores": 1, "kind": "port",
                   "variant": "dense as-written (per-call vector copies, full p x p complex products): the reference's cost profile",
                   "lean_variant_value": lean1,
                   "lean_variant": "same arithmetic in the same order (bitwise equal results), fixed-size arrays, no heap in the time loop",
                   "sample": "the full 65,536-row theta batch of one step: two passes dense + one pass lean (about 10 s), one "
                             "core, oracle/carma_oracle.cpp built -O3 -march=x86-64-v3"}
        # ---- roofline of the dominant (only) kernel of the step.  Three readings, all against the FP64 FMA peak
        # measured on this GPU in this process:
        #   frac            ALGORITHMIC flops (SURVEY 8d: Hermitian complex P, 20p^2+36p+7 per step) on the IN-PRIOR rows
        #                   only (rows outside the prior leave after the prologue and are not credited);
        #   frac_executed   FP64 flops the kernel actually executes (per-step DFMA/DMUL/DADD counts read from the SASS of
        #                   this build, profiles/r02_sass_loop_counts.json): the real-half state needs ~0.41x the
        #                   algorithmic count, so `frac` overstates how busy the pipe is;
        #   pipe_fp64_pct   sm__inst_executed_pipe_fp64 of the ncu capture of the same build (profiles/).
        counts = {}
        try:
            counts = json.load(open(os.path.join(ROOT, "profiles", "r02_sass_loop_counts.json")))["k1"][str(P)]["all_conjugate_loop"]
        except Exception:
            pass
        fin_kern_ms = in_prior["ms_per_step_rank0"]
        achieved_fin_tf = in_prior["rows_rank0"] * fe / (fin_kern_ms * 1e-3) / 1e12
        exec_flops_step = counts.get("fp64_flops")
        PROLOGUE_FP64_FLOPS = 4300.0   # ~2,500 FP64 instructions of transform_theta<5> (SASS count, FMA = 2)
        executed_tf = (in_prior["rows_rank0"] * ((NY - 1) * exec_flops_step + PROLOGUE_FP64_FLOPS) / (fin_kern_ms * 1e-3) / 1e12
                       if exec_flops_step else None)
        ncu = {}
        try:
            ncu = json.load(open(os.path.join(ROOT, "profiles", "r02_k1_ncu_summary.json")))
        except Exception:
            pass
        roofline = {
            "bound": "fp64", "achieved": achieved_fin_tf, "peak": fp64_peak, "unit": "TFLOP/s",
            "frac": achieved_fin_tf / fp64_peak if fp64_peak else None,
            "frac_definition": "algorithmic flops (SURVEY 8d) of the in-prior rows / measured FP64 FMA peak; the algorithmic "
                               "count assumes a Hermitian complex P and overstates the executed work ~2.4x",
            "achieved_all_rows": achieved_tf, "frac_all_rows": achieved_tf / fp64_peak if fp64_peak else None,
            "executed_tflops": executed_tf, "frac_executed": executed_tf / fp64_peak if (executed_tf and fp64_peak) else None,
            "executed_flops_per_step": exec_flops_step, "executed_fp64_instructions_per_step": counts.get("fp64_instructions"),
            "instructions_per_step": counts.get("instructions"),
            "dispatch_cycle_model_per_step": counts.get("dispatch_cycle_model"),
            "executed_source": "profiles/r02_sass_loop_counts.json (scripts/sass_loopstat.py on this build), all-conjugate loop, P=5",
            "pipe_fp64_pct": ncu.get("sm__inst_executed_pipe_fp64_pct"), "issue_active_pct": ncu.get("issue_active_pct"),
            "pipe_source": ncu.get("source"),
            "frac_of_datasheet": achieved_fin_tf / 40.0, "datasheet_peak": 40.0,
            "datasheet_note": "B200 vector FP64 as published (40 TFLOP/s; SURVEY 8d asks for both)",
            "traffic": ncu.get("dram_bytes_per_launch"), "traffic_source": ncu.get("traffic_source"),
            "kernel": "loglik_batch_kernel<5>", "kernel_ms": kern_ms, "kernel_ms_in_prior_rows": fin_kern_ms,
            "flops_per_eval": fe, "flops_per_step_formula": "20p^2+36p+7 (SURVEY 8d), transcendentals excluded",
            "peak_source": "DFMA saturation micro-benchmark run on this GPU in this process (carma_fp64_peak_tflops); "
                           "MEASURED_PEAKS.json has no FP64 entry; a recorded copy with clocks is profiles/FP64_PEAK.json",
            "hbm": {"achieved": alg_bytes / (kern_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                    "frac": alg_bytes / (kern_ms * 1e-3) / 1e9 / hbm_peak,
                    "algorithmic_bytes_per_launch": alg_bytes,
                    "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650"}}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": workload_config(),
            "timing": {"l2": "256 MB buffer written between timed steps (outside the event pairs)",
                       "how": "CUDA events on the launching stream, per step; sum over K steps; max over ranks"},
            "clocks": clocks,
            "e2e": {"value": world * NTHETA * K / e2e_s, "unit": UNIT, "h2d_bytes_per_step": NTHETA * d * 8,
                    "d2h_bytes_per_step": NTHETA * 8,
                    "api": "carma_loglik_batch_async/_wait: %d-slot pipeline over pinned host buffers, K steps" % NSLOT, "slots": NSLOT,
                    "h2d_gbs_this_box": h2d_gbs,
                    "repeats": E2E_REPEATS, "statistic": "median over repeats of the K-step region (max over ranks per repeat)",
                    "repeat_values": [world * NTHETA * K / x for x in pipe_s],
                    "blocking_call_value": world * NTHETA * K / e2e_block_s,
                    "blocking_api": "carma_loglik_batch (one synchronous call per step)",
                    "matches_device_path": same},
            "gpu_launches": K,
            "roofline": roofline,
            "cpu_baseline": cpu,
            "in_prior_subset": in_prior,
            "pt_mcmc": pt,
            "choose_order": order,
            "survey": survey,
            "scan": scan,
            "summary": {"max_logpost": summary[0], "finite_rows": summary[1], "checksum_rank0": checksum},
        }
        print(json.dumps(line))
        if last_out is not None:
            # rows outside the prior come back as -inf; store which rows are finite and their values, so every
            # stored number is finite and the class of each row is still compared
            fin = np.isfinite(last_out)
            os.makedirs(args.dump_outputs, exist_ok=True)
            np.save(os.path.join(args.dump_outputs, "finite_rows.npy"), fin.astype(np.float64))
            np.save(os.path.join(args.dump_outputs, "logdensity.npy"), last_out[fin])
    series.close()
    if dist:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-pt", action="store_true", help="skip the PT-MCMC secondary measurement")
    ap.add_argument("--no-cpu", action="store_true", help="skip the single-core CPU baseline")
    ap.add_argument("--no-survey", action="store_true", help="skip the multi light-curve secondary measurement")
    ap.add_argument("--no-scan", action="store_true", help="skip the ny=1e6 associative-scan measurement")
    ap.add_argument("--no-order", action="store_true", help="skip the choose_order (config 4) secondary measurement")
    ap.add_argument("--order-trials", type=int, default=100)
    ap.add_argument("--survey-curves", type=int, default=1000000, help="curves of the WHOLE survey (split over the ranks)")
    ap.add_argument("--scan-ny", type=int, default=1000000)
    ap.add_argument("--pt-ensembles", type=int, default=4096)
    ap.add_argument("--pt-iters", type=int, default=400)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps write what the last one returned for rank 0's 65,536 rows: "
                         "DIR/finite_rows.npy (1.0 where the log-density is finite, 0.0 where it is -inf outside the "
                         "prior) and DIR/logdensity.npy (the finite log-densities in row order), both float64; the "
                         "inputs are seeded, so two builds can be compared")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
