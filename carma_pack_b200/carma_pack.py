"""User-level Python API with the names and semantics of the reference's `carmcmc` package
(src/carmcmc/carma_pack.py, src/carmcmc/__init__.py:1-4), driving the GPU path.

    CarmaModel(time, y, ysig, p, q).run_mcmc(n) / .get_mle(p, q) / .choose_order(pmax)
    CarmaSample, Car1Sample: posterior container with derived quantities, predict / simulate
    get_ar_roots, power_spectrum, carma_variance, carma_process, car1_process

Out of scope (SURVEY section 2, rows 11-12): matplotlib plots and summaries.  What differs on
purpose from the reference:
  * `get_mle` / `choose_order` run all random starts of a (p,q) model in lock-step: the starting
    values come from short on-device MCMC runs (reference: carma_pack.py:199-216, one C++ MCMC run per
    trial) and the L-BFGS-B fits of the reference (carma_pack.py:250, finite-difference gradient) are
    replaced by a batched projected L-BFGS whose function and finite-difference gradient evaluations
    are single batched GPU launches;
  * CarmaSample does not re-filter the stored samples to obtain `loglik` (carma_pack.py:307-313 does, one
    FFI call per sample): with SetMLE(True) that number equals the stored log-posterior; the derived
    quantities (roots, coefficients, sigma) are vectorised numpy;
  * Python-3 bugs of the reference (SURVEY Q14) are not reproduced.
"""
import numpy as np

from . import _lib
from ._lib import (KIND_CAR1, KIND_CARP, KIND_CARMA, KIND_ZCAR, KIND_ZCARMA, IGNORE_BOUNDS, Series, model_dim)
from .synth import get_ar_roots, power_spectrum, carma_variance, carma_process, car1_process  # noqa: F401


def _kind_for(p, q):
    if p == 1:
        return KIND_CAR1
    return KIND_CARMA if q > 0 else KIND_CARP


class OptimizeResult(dict):
    """Minimal stand-in for scipy.optimize.OptimizeResult (attributes x, fun, message, success, nit, nfev)."""
    __getattr__ = dict.get
    __setattr__ = dict.__setitem__


def mle_bounds(p, q, ysigma, min_dt, tspan):
    """Box bounds of the optimiser (carma_pack.py:218-240) from the light curve's standard deviation, shortest gap and
    time span.  Scalars give (d,) arrays; arrays of curves give (..., d)."""
    ysigma, min_dt, tspan = np.broadcast_arrays(*(np.asarray(v, dtype=float) for v in (ysigma, min_dt, tspan)))
    one = np.ones_like(ysigma)
    max_freq = 0.9 / min_dt
    min_freq = 1.0 / tspan
    lo = [ysigma / 10.0, 0.9 * one, -np.inf * one]
    hi = [10.0 * ysigma, 1.1 * one, np.inf * one]
    if p == 1:
        lo.append(np.log(min_freq)); hi.append(np.log(max_freq))
    else:
        lo += [np.log(np.minimum(min_freq ** 2, 2.0 * min_freq))] * p
        hi += [np.log(np.maximum(max_freq ** 2, 2.0 * max_freq))] * p
        lo += [-np.inf * one] * q
        hi += [np.inf * one] * q
    return np.stack(lo, axis=-1), np.stack(hi, axis=-1)


def redraw_out_of_box(x0, lower, upper, seed, trials):
    """carma_pack.py:244-248 in place: every component of a row of x0 (n, d) that lies outside a finite bound is
    redrawn uniformly inside the box, by the generator of the row's global trial index, default_rng([seed % 2**63,
    trials[i]]).  lower / upper: (d,) or (n, d).  Only rows with such a component construct a generator."""
    lower = np.broadcast_to(lower, x0.shape)
    upper = np.broadcast_to(upper, x0.shape)
    out = np.isfinite(lower) & ((x0 < lower) | (x0 > upper))
    for i in np.flatnonzero(out.any(axis=1)):
        rng = np.random.default_rng([seed % (2 ** 63), int(trials[i])])
        for j in np.flatnonzero(out[i]):
            x0[i, j] = rng.uniform(lower[i, j], upper[i, j])
    return x0


def aicc(fun, p, q, ny):
    """AICc of a fit with -loglik `fun` on `ny` points (carma_pack.py:176-180), nparams = 2 + p + q as there (SURVEY Q11)."""
    nparams = 2 + p + q  # sic, carma_pack.py:178
    return 2.0 * nparams + 2.0 * fun + 2.0 * nparams * (nparams + 1.0) / (ny - nparams - 1.0)


def batched_lbfgs(fun_batch, x0, lower, upper, maxiter=1000, m=8, gtol=1e-5, ftol=2.2e-9, fd_eps=1e-8):
    """Minimise fun over a box for every row of x0 simultaneously.

    fun_batch maps an (n, d) array to n function values (non-finite values are treated as +inf).
    Projected L-BFGS with forward-difference gradients and Armijo backtracking; all rows advance in
    lock-step so that each iteration costs a few batched evaluations (n*(d+1) rows for the gradient).
    The rows share launches, nothing else: every row keeps its own (s, y) history, so its iterates do not
    depend on which other rows are in the batch.
    """
    x = np.clip(np.array(x0, dtype=float), lower, upper)
    n, d = x.shape
    big = 1e300

    def f_safe(z):
        v = np.asarray(fun_batch(z), dtype=float)
        return np.where(np.isfinite(v), v, big)

    nfev = 0

    def grad(z, fz):
        # forward differences, stepping inward at the upper bound (scipy approx_fprime epsilon = 1e-8); a component
        # whose perturbed point has no finite value is differenced the other way before it is given up
        nonlocal nfev
        h = np.full((n, d), fd_eps)
        h = np.where(z + h > upper, -h, h)
        zz = np.repeat(z[:, None, :], d, axis=1)
        idx = np.arange(d)
        zz[:, idx, idx] += h
        fv = f_safe(zz.reshape(n * d, d)).reshape(n, d)
        nfev += n * d
        g = np.where(np.abs(fv) >= big, 0.0, (fv - fz[:, None]) / h)
        bi, bj = np.nonzero(np.abs(fv) >= big)
        if bi.size:
            hb = -h[bi, bj]
            ok = (z[bi, bj] + hb >= np.broadcast_to(lower, (n, d))[bi, bj]) & (z[bi, bj] + hb <= np.broadcast_to(upper, (n, d))[bi, bj])
            pts = z[bi].copy()
            pts[np.arange(bi.size), bj] += np.where(ok, hb, 0.0)
            fb = f_safe(pts)
            nfev += bi.size
            good = ok & (np.abs(fb) < big)
            g[bi[good], bj[good]] = (fb[good] - fz[bi[good]]) / hb[good]
        return g

    f = f_safe(x)
    nfev += n
    g = grad(x, f)
    # per-row history, oldest pair first: row i holds nh[i] pairs in S[:nh[i], i] (unused entries are zero)
    S = np.zeros((m, n, d))
    Y = np.zeros((m, n, d))
    nh = np.zeros(n, dtype=int)
    restarts_left = np.full(n, 2)   # history resets granted before a row may stop on "small decrease" / failed search
    active = f < big
    nit = 0
    rows = np.arange(n)
    for nit in range(1, maxiter + 1):
        # projected gradient: zero the components pushing against an active bound
        at_lo = (x <= lower) & (g > 0)
        at_hi = (x >= upper) & (g < 0)
        pg = np.where(at_lo | at_hi, 0.0, g)
        conv = np.max(np.abs(pg), axis=1) < gtol
        active &= ~conv
        if not active.any():
            break
        # two-loop recursion, vectorised over rows; rows with fewer than h+1 pairs skip level h
        qv = pg.copy()
        alphas = [None] * m
        for h in range(m - 1, -1, -1):
            valid = h < nh
            rho = np.where(valid, 1.0 / np.maximum(np.sum(S[h] * Y[h], axis=1), 1e-300), 0.0)
            a = rho * np.sum(S[h] * qv, axis=1)
            qv -= a[:, None] * Y[h]
            alphas[h] = (a, rho)
        last = np.maximum(nh - 1, 0)
        sl, yl = S[last, rows], Y[last, rows]
        gam = np.clip(np.sum(sl * yl, axis=1) / np.maximum(np.sum(yl * yl, axis=1), 1e-300), 1e-8, 1e8)
        qv *= np.where(nh > 0, gam, 1.0 / np.maximum(np.linalg.norm(pg, axis=1), 1.0))[:, None]
        for h in range(m):
            a, rho = alphas[h]
            b = rho * np.sum(Y[h] * qv, axis=1)
            qv += (a - b)[:, None] * S[h]
        direction = -np.where(at_lo | at_hi, 0.0, qv)
        slope = np.sum(direction * pg, axis=1)
        bad = ~(slope < 0)
        direction[bad] = -pg[bad]
        slope[bad] = -np.sum(pg[bad] ** 2, axis=1)
        # batched Armijo backtracking on the projected path
        t = np.ones(n)
        xn, fn = x.copy(), f.copy()
        todo = active.copy()
        for _ in range(25):
            if not todo.any():
                break
            cand = np.clip(x + t[:, None] * direction, lower, upper)
            fc = f_safe(cand)
            nfev += n
            ok = todo & (fc <= f + 1e-4 * t * slope)
            xn[ok], fn[ok] = cand[ok], fc[ok]
            todo &= ~ok
            t[todo] *= 0.5
        moved = active & ~todo
        small = moved & ((f - fn) <= ftol * np.maximum(np.maximum(np.abs(f), np.abs(fn)), 1.0))
        gn = g.copy()
        if moved.any():
            gnew = grad(xn, fn)
            gn[moved] = gnew[moved]
        s = xn - x
        yv = gn - g
        curv = moved & (np.sum(s * yv, axis=1) > 1e-12)
        full = curv & (nh == m)
        if full.any():   # drop the oldest pair of the rows whose ring is full
            S[:-1, full] = S[1:, full]
            Y[:-1, full] = Y[1:, full]
            nh[full] -= 1
        ci = np.nonzero(curv)[0]
        S[nh[ci], ci] = s[ci]
        Y[nh[ci], ci] = yv[ci]
        nh[ci] += 1
        x, f, g = xn, fn, gn
        # line search failed or negligible decrease: drop the row's history and go on (twice at most), then stop it
        stop = (todo & active) | small
        again = stop & (nh > 0) & (restarts_left > 0)
        nh[again] = 0
        S[:, again] = 0.0
        Y[:, again] = 0.0
        restarts_left[again] -= 1
        active &= ~(stop & ~again)
    return x, f, nit, nfev


class CarmaModel(object):
    """Statistical inference assuming a CARMA(p,q) model (carma_pack.py:12-192)."""

    def __init__(self, time, y, ysig, p=1, q=0, device=0):
        if not p > q:
            raise ValueError("Order of AR polynomial, p, must be larger than order of MA polynomial, q.")
        time, y, ysig = np.asarray(time, float), np.asarray(y, float), np.asarray(ysig, float)
        # unique, ascending times (carma_pack.py:32-35)
        s_idx = np.argsort(time)
        _, u_idx = np.unique(time[s_idx], return_index=True)
        u_idx = s_idx[u_idx]
        self.time, self.y, self.ysig = time[u_idx], y[u_idx], ysig[u_idx]
        self.p, self.q = p, q
        self.device = device
        self.mcmc_sample = None
        self._series = None
        self.mle_optimizer = "device"   # "device": the fit of a start inside one kernel; "native": host loop; see get_mle

    @property
    def series(self):
        if self._series is None:
            self._series = Series(self.time, self.y, self.ysig, device=self.device)
        return self._series

    def run_mcmc(self, nsamples, nburnin=None, ntemperatures=None, nthin=1, init=None, seed=None, n_ensembles=1):
        """Run the parallel-tempering RAM sampler on the GPU (carma_pack.py:53-90).

        n_ensembles > 1 runs that many independent ensembles in the same launch and concatenates
        their coolest chains (extension; the reference runs one)."""
        p, q = self.p, self.q
        if ntemperatures is None:
            ntemperatures = max(10, p + q)
        if nburnin is None:
            nburnin = nsamples // 2
        if seed is None:
            seed = int(np.random.SeedSequence().generate_state(1, dtype=np.uint64)[0])
        kind = _kind_for(p, q)
        if p == 1:
            ntemperatures = 1  # run_mcmc_car1 has a single chain (carmcmc.cpp:30-77)
        prior = self.series.default_prior(population_var=True)  # carmcmc.cpp:85-89
        res = self.series.pt_run(kind, p, q, int(nsamples), int(nburnin), thin=int(nthin), ntemps=int(ntemperatures),
                                 n_ensembles=int(n_ensembles), seed=seed, init=init, prior=prior)
        d = model_dim(kind, p, q)
        trace = res["samples"].reshape(-1, d)
        logpost = res["logposts"].reshape(-1)
        if p == 1:
            sample = Car1Sample(self.time, self.y, self.ysig, trace=trace, logpost=logpost, series=self.series,
                                prior=prior)
        else:
            sample = CarmaSample(self.time, self.y, self.ysig, trace=trace, logpost=logpost, p=p, q=q,
                                 series=self.series, prior=prior)
        sample.accept_rates = res["accept_rates"]
        sample.exchange_rates = res["exchange_rates"]
        self.mcmc_sample = sample
        return sample

    def _mle_bounds(self, p, q):
        """Box bounds of the optimiser (carma_pack.py:218-240)."""
        return mle_bounds(p, q, self.y.std(), np.diff(self.time).min(), self.time.max() - self.time.min())

    def mle_starts(self, p, q, ntrials, seed, trial_offset=0, series=None):
        """The `ntrials` starting points of get_mle and everything that defines the fits: (kind, x0, lower, upper,
        prior, flags).  Start j depends only on (seed, trial_offset + j): short on-device MCMC runs with nsamples=1,
        nburnin=25, nwalkers=10 as in the reference (carma_pack.py:197-216), measerr_scale set to 1 (:216), components
        outside the optimiser's box redrawn uniformly inside it (:244-248)."""
        series = self.series if series is None else series
        kind = _kind_for(p, q)
        d = model_dim(kind, p, q)
        prior = series.default_prior(population_var=True)
        res = series.pt_run(kind, p, q, 1, 25, ntemps=1 if p == 1 else 10, n_ensembles=ntrials, seed=seed,
                            ensemble_offset=trial_offset, prior=prior)
        x0 = res["samples"][:, 0, :].copy()
        x0[:, 1] = 1.0  # carma_pack.py:216
        lo, hi = self._mle_bounds(p, q)
        redraw_out_of_box(x0, lo, hi, seed, trial_offset + np.arange(ntrials))
        flags = 0 if p == 1 else IGNORE_BOUNDS  # SetMLE(True) only for p > 1 (carma_pack.py:242)
        return kind, x0, lo, hi, prior, flags

    def get_mle(self, p, q, ntrials=100, njobs=1, seed=None, maxiter=1000, trial_offset=0, series=None,
                optimizer=None):
        """Maximum-likelihood estimate from `ntrials` random starts (carma_pack.py:92-129), all trials
        in lock-step on the GPU.  `njobs` is accepted for API compatibility and ignored.  trial_offset:
        global index of the first trial (multi-GPU sharding: the starts of trial j do not depend on which
        rank runs it).  series: device series to use (choose_order gives each worker thread its own).
        optimizer: "device" = carma_mle_batch_device (the whole fit inside one kernel, one warp per start);
        "native" = carma_mle_batch (C++ host loop, one launch per batch of trial points);
        "python" = the same algorithm in numpy (batched_lbfgs), kept as the cross-check.  None: self.mle_optimizer."""
        series = self.series if series is None else series
        if seed is None:
            seed = int(np.random.SeedSequence().generate_state(1, dtype=np.uint64)[0])
        kind, x0, lo, hi, prior, flags = self.mle_starts(p, q, ntrials, seed, trial_offset=trial_offset, series=series)

        def negloglik(th):  # _carma_loglik, carma_pack.py:255-260
            # through the slot API: its own stream, so concurrent fits of other models overlap on the GPU
            th = np.ascontiguousarray(th, dtype=np.float64)
            out = np.empty(th.shape[0])
            series.loglik_async(kind, p, q, th.ctypes.data, out.ctypes.data, th.shape[0], prior, 0, flags=flags)
            series.loglik_wait(0)
            return -out

        if optimizer is None:
            optimizer = self.mle_optimizer
        if optimizer in ("native", "device"):
            x, f, nit, nfev = series.mle_batch(kind, p, q, x0, lo, hi, prior=prior, flags=flags, maxiter=maxiter,
                                               on_device=(optimizer == "device"))
        elif optimizer == "python":
            x, f, nit, nfev = batched_lbfgs(negloglik, x0, lo, hi, maxiter=maxiter)
        else:
            raise ValueError("optimizer must be 'device', 'native' or 'python'")
        return self._mle_result(x, f, nit, nfev)

    def hessian(self, theta, p=None, q=None, rel_step=None):
        """Gradient, Hessian and Laplace covariance of the log-density at theta (e.g. get_mle(...).x), with get_mle's
        model kind, population-variance prior and flags: MultiSeries.hessian on this curve alone, so it equals a survey
        row bit for bit.  Returns loglik (scalar), grad (d,), hessian (d, d), cov (d, d), stderr (d,), status, step (d,)."""
        p = self.p if p is None else p
        q = self.q if q is None else q
        ms = _lib.MultiSeries(self.time, self.y, self.ysig, [0, self.time.size], device=self.device)
        try:
            res = ms.hessian(_kind_for(p, q), p, q, np.asarray(theta, dtype=np.float64)[None, :], rel_step=rel_step)
        finally:
            ms.close()
        return OptimizeResult({k: (v[0].item() if v.ndim == 1 else v[0]) for k, v in res.items()})

    def laplace_sample(self, theta, p=None, q=None, cov=None, ndraws=1000, seed=None):
        """The posterior by importance sampling from the Laplace approximation at theta (e.g. get_mle(...).x):
        MultiSeries.laplace_sample on this curve alone (curve_offset 0), so it equals a one-curve survey call bit for bit.
        cov None: the covariance of self.hessian(theta).  Returns a CarmaSample (Car1Sample for p = 1) of the resampled
        draws, carrying khat, ess and status (k-hat above 0.7: the Gaussian proposal misses the posterior; run_mcmc)."""
        p = self.p if p is None else p
        q = self.q if q is None else q
        if seed is None:
            seed = int(np.random.SeedSequence().generate_state(1, dtype=np.uint64)[0] >> 1)
        th = np.asarray(theta, dtype=np.float64)[None, :]
        cv = None if cov is None else np.asarray(cov, dtype=np.float64)[None, :, :]
        ms = _lib.MultiSeries(self.time, self.y, self.ysig, [0, self.time.size], device=self.device)
        try:
            ls = ms.laplace_sample(p, q, th, cov=cv, ndraws=ndraws, seed=seed)
        finally:
            ms.close()
        prior = self.series.default_prior(population_var=True)
        if p == 1:
            sample = Car1Sample(self.time, self.y, self.ysig, trace=ls.trace[0], logpost=ls.logpost[0], series=self.series,
                                prior=prior)
        else:
            sample = CarmaSample(self.time, self.y, self.ysig, trace=ls.trace[0], logpost=ls.logpost[0], p=p, q=q,
                                 series=self.series, prior=prior)
        sample.khat, sample.ess, sample.status = float(ls.khat[0]), float(ls.ess[0]), int(ls.status[0])
        return sample

    @staticmethod
    def _mle_result(x, f, nit, nfev):
        best = int(np.argmin(f))
        return OptimizeResult(x=x[best], fun=float(f[best]), nit=nit, nfev=nfev, success=bool(np.isfinite(f[best])),
                              message="batched projected L-BFGS, best of %d starts" % len(f), all_x=x, all_fun=f)

    def choose_order(self, pmax, qmax=None, pqlist=None, njobs=1, ntrials=100, seed=None, verbose=True, dist=None):
        """Choose (p,q) by minimising AICc over a grid of MLEs (carma_pack.py:131-192).

        dist: an initialised torch.distributed module (one process per GPU).  The (p,q) models are then
        partitioned over the ranks by cost (sharding.partition_weighted) and only the per-model summaries
        (AICc, -loglik, theta-hat) are all-gathered; every rank returns the same result."""
        if not pmax > 0:
            raise ValueError("Order of AR polynomial must be at least 1.")
        if qmax is None:
            qmax = pmax - 1
        if not pmax > qmax:
            raise ValueError("Order of AR polynomial, p, must be larger than order of MA polynimial, q.")
        if pqlist is None:
            pqlist = [(p, q) for p in range(1, pmax + 1) for q in range(min(p, qmax + 1))]
        world = 1
        units = [(k, 0, ntrials) for k in range(len(pqlist))]   # (model, first trial, number of trials)
        if dist is not None and dist.is_initialized() and dist.get_world_size() > 1:
            from . import sharding
            world = dist.get_world_size()
            # unit of work = one (model, trial); cost ~ F_step(p) (d+1); contiguous cost-weighted blocks
            cost1 = [(20 * p * p + 36 * p + 7) * (4 + p + q) for p, q in pqlist]
            costs = np.repeat(np.array(cost1, dtype=float), ntrials)
            mine = sharding.partition_weighted(costs, world, dist.get_rank())
            units = []
            for k in sorted(set(int(u) // ntrials for u in mine)):
                tr = [int(u) % ntrials for u in mine if int(u) // ntrials == k]
                units.append((k, min(tr), len(tr)))
        # The fits of different (p,q) models are independent and each one is a chain of small, latency-bound
        # launches: run several of them concurrently from worker threads, each with its own device series
        # (own scratch buffers and stream), so their launches overlap on the GPU.  Heaviest models first.
        from concurrent.futures import ThreadPoolExecutor
        units.sort(key=lambda u: -(pqlist[u[0]][0] ** 2) * (4 + sum(pqlist[u[0]])) * u[2])
        # the fits release the GIL; each worker spins in a stream synchronise while its launch runs, so more
        # workers than host cores only add contention
        import os
        nworkers = max(1, min(len(units), max(4, min(16, os.cpu_count() or 8))))
        if os.environ.get("CARMA_ORDER_WORKERS"):
            nworkers = max(1, min(len(units), int(os.environ["CARMA_ORDER_WORKERS"])))
        pool_series = [Series(self.time, self.y, self.ysig, device=self.device) for _ in range(nworkers)]
        import queue
        free = queue.Queue()
        for srs in pool_series:
            free.put(srs)

        if seed is None:
            seed = int(np.random.SeedSequence().generate_state(1, dtype=np.uint64)[0]) % (2 ** 62)

        def fit(unit):
            k, first, count = unit
            p, q = pqlist[k]
            srs = free.get()
            try:
                if self.mle_optimizer == "device":   # only the starting values here (short runs), the fits below
                    return k, self.mle_starts(p, q, count, seed + k, trial_offset=first, series=srs)
                return k, self.get_mle(p, q, ntrials=count, njobs=njobs, seed=seed + k, trial_offset=first, series=srs)
            finally:
                free.put(srs)

        with ThreadPoolExecutor(max_workers=nworkers) as ex:
            local = dict(ex.map(fit, units))
        if self.mle_optimizer == "device":
            # every start of every model in ONE launch (carma_mle_grid_device): the device serves them from a queue,
            # heaviest model first; separate launches per model do not overlap well (see mle_dev.cu)
            ks = [u[0] for u in units]
            fits = pool_series[0].mle_grid([(local[k][0],) + tuple(pqlist[k]) + tuple(local[k][1:]) for k in ks])
            local = {k: self._mle_result(*r) for k, r in zip(ks, fits)}
        for srs in pool_series:
            srs.close()
        if world > 1:
            from . import sharding
            dmax = max(3 + p + q for p, q in pqlist)
            # row = [-loglik (selection key), nit, nfev, theta-hat..., nan padding]
            table = np.full((len(pqlist), 3 + dmax), np.nan)
            table[:, 0] = np.inf
            for k, mle in local.items():
                table[k, 0], table[k, 1], table[k, 2] = mle.fun, mle.nit, mle.nfev
                table[k, 3:3 + len(mle.x)] = mle.x
            best = sharding.best_per_model(table, dist)
            MLEs = []
            for k, (p, q) in enumerate(pqlist):
                d = 4 if p == 1 else 3 + p + q
                MLEs.append(OptimizeResult(x=best[k, 3:3 + d].copy(), fun=float(best[k, 0]), nit=int(best[k, 1]),
                                           nfev=int(best[k, 2]), success=bool(np.isfinite(best[k, 0])),
                                           message="batched projected L-BFGS, best over all ranks' starts (all_x / all_fun "
                                                   "stay on the rank that ran them)"))
        else:
            MLEs = [local[k] for k in range(len(pqlist))]
        best_AICc, AICc, best_MLE = 1e300, [], MLEs[0]
        if verbose:
            print("p, q, AICc:")
        for MLE, (p, q) in zip(MLEs, pqlist):
            this_AICc = aicc(MLE.fun, p, q, self.time.size)
            if verbose:
                print(p, q, this_AICc)
            AICc.append(this_AICc)
            if this_AICc < best_AICc:
                best_MLE, best_AICc = MLE, this_AICc
                self.p, self.q = p, q
        if verbose:
            print("Model with best AICc has p =", self.p, " and q = ", self.q)
        return best_MLE, pqlist, AICc


def _survey_starts(ms, p, q, ntrials, seed, curve_offset, priors, stats):
    """CarmaModel.mle_starts for every curve of the multi-series `ms`: one multi-curve PT launch (ensemble of curve c,
    trial j = global trial (curve_offset + c) * ntrials + j), measerr_scale := 1, out-of-box components redrawn.
    Returns (kind, x0 (ncurves, ntrials, d), lower (ncurves, d), upper (ncurves, d), flags)."""
    kind = _kind_for(p, q)
    d = model_dim(kind, p, q)
    nc = ms.ncurves
    res = ms.pt_run(kind, p, q, 1, 25, ntemps=1 if p == 1 else 10, n_ensembles=ntrials, seed=seed,
                    ensemble_offset=curve_offset * ntrials, priors=priors)
    x0 = np.ascontiguousarray(res["samples"][:, :, 0, :])
    x0[:, :, 1] = 1.0  # carma_pack.py:216
    lo, hi = mle_bounds(p, q, np.sqrt(stats["y_var_pop"]), stats["min_dt"], stats["tspan"])
    trials = (curve_offset + np.arange(nc))[:, None] * ntrials + np.arange(ntrials)[None, :]
    redraw_out_of_box(x0.reshape(nc * ntrials, d), np.repeat(lo, ntrials, axis=0), np.repeat(hi, ntrials, axis=0), seed,
                      trials.reshape(-1))
    flags = 0 if p == 1 else IGNORE_BOUNDS  # SetMLE(True) only for p > 1 (carma_pack.py:242)
    return kind, x0, lo, hi, flags


def _survey_result(x, f, nit, nfev, x0, lo, hi):
    best = np.argmin(f, axis=1)
    rows = np.arange(f.shape[0])
    fun = f[rows, best]
    return OptimizeResult(x=x[rows, best], fun=fun, nit=nit, nfev=nfev, success=np.isfinite(fun),
                          message="batched projected L-BFGS, best of %d starts per curve" % f.shape[1],
                          all_x=x, all_fun=f, x0=x0, lower=lo, upper=hi)


def _random_seed():
    return int(np.random.SeedSequence().generate_state(1, dtype=np.uint64)[0]) % (2 ** 62)


def survey_get_mle(ms, p, q, ntrials=100, seed=None, maxiter=1000, curve_offset=0, priors=None):
    """CarmaModel.get_mle for every light curve of the multi-series `ms` (MultiSeries.get_mle): starting values of all
    curves from one PT launch, then the fits of all curves x starts in one launch.  Returns an OptimizeResult of
    per-curve arrays: x (ncurves, d) best of the starts, fun, nit, nfev, success, all_x (ncurves, ntrials, d), all_fun,
    and the x0 / lower / upper rows the fits used."""
    if not p > q:
        raise ValueError("Order of AR polynomial, p, must be larger than order of MA polynomial, q.")
    if seed is None:
        seed = _random_seed()
    stats = ms.curve_stats()
    kind, x0, lo, hi, flags = _survey_starts(ms, p, q, ntrials, seed, curve_offset, priors, stats)
    (x, f, nit, nfev), = ms.mle_grid([(kind, p, q, x0, lo, hi, flags)], priors=priors, maxiter=maxiter)
    return _survey_result(x, f, nit, nfev, x0, lo, hi)


def survey_choose_order(ms, pmax, qmax=None, pqlist=None, ntrials=100, seed=None, curve_offset=0):
    """CarmaModel.choose_order for every light curve of the multi-series `ms` (MultiSeries.choose_order): the same
    default grid and seeds (model k uses seed + k), one starting-value launch per model, then ONE launch fitting every
    model on every curve from every start.  Per-curve AICc with the reference's formula and each curve's own ny.
    Returns (best_pq (ncurves, 2), pqlist, aicc (ncurves, nmodels), mles) with mles[k] model k's per-curve result."""
    if not pmax > 0:
        raise ValueError("Order of AR polynomial must be at least 1.")
    if qmax is None:
        qmax = pmax - 1
    if not pmax > qmax:
        raise ValueError("Order of AR polynomial, p, must be larger than order of MA polynimial, q.")
    if pqlist is None:
        pqlist = [(p, q) for p in range(1, pmax + 1) for q in range(min(p, qmax + 1))]
    if seed is None:
        seed = _random_seed()
    stats = ms.curve_stats()
    starts = [_survey_starts(ms, p, q, ntrials, seed + k, curve_offset, None, stats) for k, (p, q) in enumerate(pqlist)]
    fits = ms.mle_grid([(kind, p, q, x0, lo, hi, flags)
                        for (kind, x0, lo, hi, flags), (p, q) in zip(starts, pqlist)])
    mles = [_survey_result(x, f, nit, nfev, st[1], st[2], st[3]) for (x, f, nit, nfev), st in zip(fits, starts)]
    table = np.stack([aicc(mle.fun, p, q, stats["ny"]) for mle, (p, q) in zip(mles, pqlist)], axis=1)
    best = np.argmin(table, axis=1)
    best_pq = np.asarray(pqlist, dtype=int)[best]
    return best_pq, pqlist, table, mles


def survey_run_mcmc(ms, p, q, nsamples, nburnin=None, ntemperatures=None, nthin=1, seed=None, n_ensembles=1, priors=None):
    """CarmaModel.run_mcmc for every light curve of the multi-series `ms` (MultiSeries.run_mcmc): the same defaults
    (ntemperatures = max(10, p + q), one chain for p = 1, nburnin = nsamples // 2, population-variance priors), all
    curves in one carma_multi_pt_run launch.  Returns a SurveySample."""
    if not p > q:
        raise ValueError("Order of AR polynomial, p, must be larger than order of MA polynomial, q.")
    if ntemperatures is None:
        ntemperatures = max(10, p + q)
    if nburnin is None:
        nburnin = nsamples // 2
    if seed is None:
        seed = int(np.random.SeedSequence().generate_state(1, dtype=np.uint64)[0])
    if p == 1:
        ntemperatures = 1  # run_mcmc_car1 has a single chain (carmcmc.cpp:30-77)
    kind = _kind_for(p, q)
    if priors is None:
        priors = ms.default_priors(population_var=True)  # carmcmc.cpp:85-89
    res = ms.pt_run(kind, p, q, int(nsamples), int(nburnin), thin=int(nthin), ntemps=int(ntemperatures),
                    n_ensembles=int(n_ensembles), seed=seed, priors=priors)
    nc, d = ms.ncurves, model_dim(kind, p, q)
    sample = SurveySample(res["samples"].reshape(nc, -1, d), res["logposts"].reshape(nc, -1), p, q, kind=kind,
                          priors=priors, stats=ms.curve_stats(), multi_series=ms)
    sample.accept_rates = res["accept_rates"]
    sample.exchange_rates = res["exchange_rates"]
    return sample


class SurveySample(object):
    """The posterior samples of every curve of a survey (MultiSeries.run_mcmc): what CarmaSample / Car1Sample give for
    one curve, as per-curve arrays.  trace (ncurves, nsamples, d) with the ensembles of a curve one after the other, as
    CarmaModel.run_mcmc concatenates them; logpost (ncurves, nsamples).  Derived parameters come from one device launch
    over the whole trace, made when one is first asked for; the power-spectrum band and the effective sample sizes run
    on the device without the per-sample arrays crossing PCIe.  stats: MultiSeries.curve_stats() (the default frequency
    grid); priors: PRIOR_DTYPE per curve; multi_series: the survey the trace came from (for curve())."""

    _DERIVED = ("ar_roots", "psd_width", "psd_centroid", "ar_coefs", "ma_coefs", "sigma")

    def __init__(self, trace, logpost, p, q, kind=None, priors=None, stats=None, multi_series=None):
        self.trace = np.asarray(trace, dtype=float)
        self.logpost = np.asarray(logpost, dtype=float)
        if self.trace.ndim != 3 or self.logpost.shape != self.trace.shape[:2]:
            raise ValueError("trace must be (ncurves, nsamples, d) and logpost (ncurves, nsamples)")
        self.p, self.q = p, q
        self.kind = _kind_for(p, q) if kind is None else kind
        if self.trace.shape[2] != model_dim(self.kind, p, q):
            raise ValueError("trace rows must have %d entries for this model" % model_dim(self.kind, p, q))
        self.ncurves, self.nsamples = self.trace.shape[:2]
        self.priors, self.stats, self.multi_series = priors, stats, multi_series
        self._derived = None

    def _prior_struct(self, c):
        return None if self.priors is None else _lib.Prior(*[float(v) for v in self.priors[c]])

    def _derive(self):
        if self._derived is None:
            if self.kind == KIND_ZCARMA:
                raise ValueError("derived parameters of a ZCARMA survey need per-curve kappa bounds; use curve()")
            der = _lib.derived_params(self.kind, self.p, self.q, self.trace.reshape(-1, self.trace.shape[2]))
            shape = (self.ncurves, self.nsamples)
            self._derived = {k: v.reshape(shape + v.shape[1:]) for k, v in der.items()}
            self._derived["ma_coefs"] = self._derived["ma_coefs"][:, :, :self.q + 1]
        return self._derived

    def get_samples(self, name):
        """The CarmaSample / Car1Sample entry `name` of every curve: (ncurves, nsamples) for scalars, (ncurves,
        nsamples, k) for vectors."""
        th = self.trace
        if name == "var":
            return th[:, :, 0] ** 2
        if name == "measerr_scale":
            return th[:, :, 1].copy()
        if name == "mu":
            return th[:, :, 2].copy()
        if name in ("loglik", "logpost"):
            return self.logpost.copy()
        if name == "loglik_only":
            return self.logpost - CarmaSample.log_prior(th.reshape(-1, th.shape[2])).reshape(self.logpost.shape)
        if self.p == 1 and self.kind == KIND_CAR1:
            if name == "log_omega":
                return th[:, :, 3].copy()
            if name == "sigma":   # Car1Sample: sqrt(2 omega var)
                return np.sqrt(2.0 * np.exp(th[:, :, 3]) * th[:, :, 0] ** 2)
        elif name == "quad_coefs":
            return np.exp(th[:, :, 3:3 + self.p])
        if name in self._DERIVED and not (self.kind == KIND_CAR1 and name in ("ar_coefs", "ma_coefs")):
            return self._derive()[name].copy()
        raise KeyError(name)

    def best_index(self):
        """Index of the largest log-posterior of every curve (ncurves,): CarmaSample.best_index per curve."""
        return np.argmax(self.logpost, axis=1)

    def map_theta(self):
        """The maximum-a-posteriori theta row of every curve (ncurves, d), the input of MultiSeries.predict /
        kalman_filter / conditional_simulate."""
        return self.trace[np.arange(self.ncurves), self.best_index()].copy()

    def DIC(self):
        """CarmaSample.DIC of every curve (ncurves,) (carma_pack.py:808-828)."""
        ll = self.logpost
        return -2.0 * ll.mean(axis=1) + 2.0 * np.var(-2.0 * ll, axis=1) / 2.0

    def effective_samples(self, name):
        """MCMCSample.effective_samples of `name` (a real-valued entry) for every curve, on the device: (ncurves, k)."""
        x = np.asarray(self.get_samples(name))
        if np.iscomplexobj(x):
            raise ValueError("effective_samples needs a real-valued entry, %r is complex" % name)
        if x.ndim == 2:
            x = x[:, :, None]
        return _lib.effective_samples(x)

    def default_freq(self):
        """CarmaSample's frequency grid of every curve (ncurves, 200): 200 log-spaced points from 1 / tspan to
        0.5 / min_dt."""
        if self.stats is None:
            raise ValueError("the default frequency grid needs the curve statistics (MultiSeries.curve_stats())")
        lo = np.log10(1.0 / np.asarray(self.stats["tspan"], dtype=float))
        hi = np.log10(0.5 / np.asarray(self.stats["min_dt"], dtype=float))
        return np.stack([np.logspace(a, b, 200) for a, b in zip(lo, hi)])

    def psd_credible_band(self, percentile=68.0, freq=None):
        """CarmaSample.psd_credible_band of every curve over all its samples (slice the trace for a subset), on the
        device (carma_psd_quantiles).  freq: None (CarmaSample's grid per curve), (nfreq,) or (ncurves, nfreq).
        Returns (psd_lo, psd_hi, psd_mid, freq), each (ncurves, nfreq)."""
        freq = self.default_freq() if freq is None else np.asarray(freq, dtype=float)
        lo, hi = (100.0 - percentile) / 2.0, 100.0 - (100.0 - percentile) / 2.0
        out = _lib.psd_quantiles(self.kind, self.p, self.q, self.trace, freq, [lo, hi, 50.0], priors=self.priors)
        freq = np.broadcast_to(freq, (self.ncurves, freq.shape[-1])).copy()
        return out[:, 0], out[:, 1], out[:, 2], freq

    def curve(self, c):
        """The CarmaSample (Car1Sample for p = 1) of curve c, built from the same arrays: the bridge to per-curve code."""
        if self.multi_series is None:
            raise ValueError("curve() needs the multi-series the samples came from")
        t, y, e = self.multi_series.curve(c)
        if self.kind == KIND_CAR1:
            return Car1Sample(t, y, e, trace=self.trace[c], logpost=self.logpost[c], prior=self._prior_struct(c))
        return CarmaSample(t, y, e, trace=self.trace[c], logpost=self.logpost[c], p=self.p, q=self.q,
                           prior=self._prior_struct(c))


class LaplaceSample(SurveySample):
    """The posterior samples of every curve of a survey by importance sampling from its Laplace approximation
    (MultiSeries.laplace_sample): trace (ncurves, ndraws, d) the equally weighted resample of the draws, logpost their
    log-posteriors; NaN rows for a curve whose status is not LAPLACE_OK.  khat (ncurves,): the Pareto k-hat of the
    weights, the reliability of the sample (<= 0.7: use it; above: run MCMC on that curve); ess (ncurves,) the weight
    ESS; status (ncurves,); laplace: the raw MultiSeries.laplace result (draws, weights, resample indices)."""

    def __init__(self, trace, logpost, p, q, laplace, kind=None, priors=None, stats=None, multi_series=None):
        super(LaplaceSample, self).__init__(trace, logpost, p, q, kind=kind, priors=priors, stats=stats,
                                            multi_series=multi_series)
        self.laplace = laplace
        self.khat, self.ess, self.status = laplace.khat, laplace.ess, laplace.status

    def effective_samples(self, name):
        raise ValueError("the draws of a LaplaceSample are resampled, not a chain: autocorrelation ESS means nothing "
                         "for them; .ess holds each curve's weight ESS")


class MCMCSample(object):
    """Dictionary of traces (subset of src/carmcmc/samplers.py:13-408 without the plots)."""

    def __init__(self, trace=None, logpost=None):
        self._samples = {}
        if logpost is not None:
            self._samples["logpost"] = np.asarray(logpost)
        self.parameters = []

    def get_samples(self, name):
        return self._samples[name].copy()

    def newaxis(self):
        for k, v in self._samples.items():
            if v.ndim == 1:
                self._samples[k] = v[:, np.newaxis]

    def effective_samples(self, name):
        """Integrated-autocorrelation estimate of the effective sample size (samplers.py uses `acor`)."""
        x = np.atleast_2d(self._samples[name].T)
        out = []
        for row in x:
            r = row - row.mean()
            n = r.size
            ac = np.correlate(r, r, mode="full")[n - 1:] / max(np.dot(r, r), 1e-300)
            tau, k = 1.0, 1
            while k < n and ac[k] > 0.05:
                tau += 2.0 * ac[k]
                k += 1
            out.append(n / tau)
        return np.array(out)


class CarmaSample(MCMCSample):
    """MCMC samples of a CARMA(p,q) model with derived quantities (carma_pack.py:263-546)."""

    def __init__(self, time, y, ysig, sampler=None, q=0, filename=None, MLE=None, trace=None, logpost=None, p=None,
                 series=None, prior=None, postprocess="device"):
        """Reference signature (carma_pack.py:267): CarmaSample(time, y, ysig, sampler, q=0, filename=None,
        MLE=None) with `sampler` the object returned by run_mcmc_carma.  Alternatively pass trace/logpost
        arrays.  postprocess: "device" (default) derives roots / coefficients / sigma of every sample in one kernel
        launch (carma_derived_params); "numpy" is the vectorised host twin kept as the cross-check (and for the
        tests that run without a GPU).  As in the reference, p is taken from the trace width minus 3 minus q (so a caller that
        forgets q gets p = p_true + q_true, which the reference's own test relies on: testCarmcmc.py:96)."""
        if sampler is not None:
            trace = np.array([list(r) for r in sampler.getSamples()], dtype=float)
            logpost = np.array(list(sampler.GetLogLikes()), dtype=float)
        if trace is None or logpost is None:
            raise ValueError("CarmaSample needs either a sampler object or trace and logpost arrays")
        trace = np.asarray(trace, dtype=float)
        logpost = np.asarray(logpost, dtype=float)
        if p is None:
            p = trace.shape[1] - 3 - q
        super(CarmaSample, self).__init__(trace=trace, logpost=logpost)
        time, y, ysig = np.asarray(time, float), np.asarray(y, float), np.asarray(ysig, float)
        self.time, self.y, self.ysig = time, y, ysig
        self.p, self.q = p, q
        self._series_obj = series      # created on first use (predict / simulate / kalman_filter): the
        self._prior_obj = prior        # post-processing below needs no GPU
        # column names as samplers.py / carma_pack.py:286-305
        self._samples["var"] = trace[:, 0] ** 2
        self._samples["measerr_scale"] = trace[:, 1]
        self._samples["mu"] = trace[:, 2]
        self._samples["quad_coefs"] = np.exp(trace[:, 3:3 + p])
        self._trace = trace
        if postprocess == "device":
            self._derive_on_device(trace)
        elif postprocess == "numpy":
            self._ar_roots()
            self._ar_coefs()
            self._ma_coefs(trace)
            self._sigma_noise()
        else:
            raise ValueError("postprocess must be 'device' or 'numpy'")
        # "loglik" of the reference = getLogDensity with SetMLE(True) for every stored sample: nsamples more filter runs
        # across the FFI (carma_pack.py:307-313).  SetMLE(True) only skips the prior-BOUNDS test; LogPrior is still added
        # (carpack.hpp:173, 180; SURVEY Q2), and every stored sample lies inside the bounds, so that number IS the stored
        # log-posterior: nothing is re-filtered.  The pure log-likelihood (log-posterior minus LogPrior) is offered next
        # to it as "loglik_only".
        self._samples["loglik"] = logpost.copy()
        self._samples["loglik_only"] = logpost - self.log_prior(trace)
        self.parameters = list(self._samples.keys())
        self.newaxis()
        self.mle = {}
        if MLE is not None:
            self.add_mle(MLE)

    @property
    def _series(self):
        if self._series_obj is None:
            self._series_obj = Series(self.time, self.y, self.ysig)
        return self._series_obj

    @property
    def _prior(self):
        if self._prior_obj is None:
            self._prior_obj = self._series.default_prior(True)
        return self._prior_obj

    @staticmethod
    def log_prior(trace, measerr_dof=50.0):
        """CARMA_Base::LogPrior (carpack.hpp:118-126) for every row: the scaled inverse-chi^2 prior on measerr_scale."""
        scale = np.asarray(trace, dtype=float)[:, 1]
        return -0.5 * measerr_dof / scale - (1.0 + measerr_dof / 2.0) * np.log(scale)

    def recompute_loglik(self):
        """The reference's loop (carma_pack.py:307-313) as ONE batched launch: LogDensity with SetMLE(True) of every
        stored sample.  Only needed to audit the stored log-posteriors; CarmaSample itself does not call it."""
        kind = KIND_CARMA if self.q > 0 else KIND_CARP
        return self._series.loglik(kind, self.p, self.q, self._trace, prior=self._prior, flags=IGNORE_BOUNDS)

    def _derive_on_device(self, trace):
        """carma_pack.py:439-546 for all samples at once on the GPU: same dictionary entries as the numpy twin below."""
        kind = KIND_CARMA if self.q > 0 else KIND_CARP
        der = _lib.derived_params(kind, self.p, self.q, trace)
        self._samples["ar_roots"] = der["ar_roots"]
        self._samples["psd_width"] = der["psd_width"]
        self._samples["psd_centroid"] = der["psd_centroid"]
        self._samples["ar_coefs"] = der["ar_coefs"]
        self._samples["ma_coefs"] = der["ma_coefs"][:, :self.q + 1]
        self._samples["sigma"] = der["sigma"]

    def _ar_roots(self):  # carma_pack.py:439-467
        qc = self._samples["quad_coefs"]
        n, p = qc.shape[0], self.p
        roots = np.empty((n, p), dtype=complex)
        for i in range(p // 2):
            q1, q2 = qc[:, 2 * i], qc[:, 2 * i + 1]
            disc = q2 ** 2 - 4.0 * q1
            sq = np.where(disc > 0, np.sqrt(np.abs(disc)), 1j * np.sqrt(np.abs(disc)))
            roots[:, 2 * i] = -0.5 * (q2 + sq)
            roots[:, 2 * i + 1] = -0.5 * (q2 - sq)
        if p % 2 == 1:
            roots[:, -1] = -qc[:, -1]
        self._samples["ar_roots"] = roots
        self._samples["psd_width"] = -roots.real / (2.0 * np.pi)
        self._samples["psd_centroid"] = np.abs(roots.imag) / (2.0 * np.pi)

    @staticmethod
    def _poly_from_roots(roots):
        """Row-wise np.poly (coefficients of prod (x - r_k), highest order first), vectorised over samples."""
        n, k = roots.shape
        coefs = np.zeros((n, k + 1), dtype=complex)
        coefs[:, 0] = 1.0
        for i in range(k):
            coefs[:, 1:i + 2] = coefs[:, 1:i + 2] - roots[:, i:i + 1] * coefs[:, 0:i + 1]
        return coefs

    def _ar_coefs(self):  # carma_pack.py:500-509
        self._samples["ar_coefs"] = self._poly_from_roots(self._samples["ar_roots"]).real

    def _ma_coefs(self, trace):  # carma_pack.py:469-498
        n = trace.shape[0]
        if self.q == 0:
            self._samples["ma_coefs"] = np.ones((n, 1))
            return
        qc = np.exp(trace[:, 3 + self.p:3 + self.p + self.q])
        roots = np.empty(qc.shape, dtype=complex)
        for i in range(self.q // 2):
            q1, q2 = qc[:, 2 * i], qc[:, 2 * i + 1]
            disc = q2 ** 2 - 4.0 * q1
            sq = np.where(disc > 0, np.sqrt(np.abs(disc)), 1j * np.sqrt(np.abs(disc)))
            roots[:, 2 * i] = -0.5 * (q2 + sq)
            roots[:, 2 * i + 1] = -0.5 * (q2 - sq)
        if self.q % 2 == 1:
            roots[:, -1] = -qc[:, -1]
        c = self._poly_from_roots(roots)
        self._samples["ma_coefs"] = (c / c[:, self.q:self.q + 1])[:, ::-1].real

    def _sigma_noise(self):  # carma_pack.py:511-546
        var, roots, ma = self._samples["var"], self._samples["ar_roots"], self._samples["ma_coefs"]
        total = np.zeros(var.shape[0], dtype=complex)
        for k in range(self.p):
            denom = -2.0 * roots[:, k].real + 0j
            for l in range(self.p):
                if l != k:
                    denom = denom * (roots[:, l] - roots[:, k]) * (np.conjugate(roots[:, l]) + roots[:, k])
            s1 = np.zeros(var.shape[0], dtype=complex)
            s2 = np.zeros(var.shape[0], dtype=complex)
            for l in range(ma.shape[1]):
                s1 += ma[:, l] * roots[:, k] ** l
                s2 += ma[:, l] * (-roots[:, k]) ** l
            total += s1 * s2 / denom
        self._samples["sigma"] = np.sqrt(var / total.real)

    def add_mle(self, MLE):  # carma_pack.py:331-405 (values only)
        th = np.asarray(MLE.x)[None, :]
        tmp = CarmaSample.__new__(CarmaSample)
        MCMCSample.__init__(tmp)
        tmp.p, tmp.q = self.p, self.q
        tmp._samples = {"var": th[:, 0] ** 2, "measerr_scale": th[:, 1], "mu": th[:, 2],
                        "quad_coefs": np.exp(th[:, 3:3 + self.p])}
        tmp._ar_roots(); tmp._ar_coefs(); tmp._ma_coefs(th); tmp._sigma_noise()
        self.mle = {k: v[0] for k, v in tmp._samples.items()}
        self.mle["loglik"] = -MLE.fun

    def _params_at(self, index):
        roots = self._samples["ar_roots"][index]
        ma = np.zeros(self.p)
        mc = self._samples["ma_coefs"][index]
        ma[:mc.size] = mc
        sigsqr = float(np.ravel(self._samples["sigma"][index])[0]) ** 2
        mu = float(np.ravel(self._samples["mu"][index])[0])
        scale = float(np.ravel(self._samples["measerr_scale"][index])[0])
        return sigsqr, roots, ma, mu, scale

    def best_index(self):
        return int(np.argmax(np.ravel(self._samples["logpost"])))

    def predict(self, time, bestfit="map"):
        """Expected value and variance of the light curve at `time` given the data (carma_pack.py:746-806):
        all query times in one launch (KalmanFilterp::Predict, one GPU thread per time)."""
        idx = self.best_index() if bestfit == "map" else int(bestfit)
        sigsqr, roots, ma, mu, scale = self._params_at(idx)
        qm, qv = self._series.predict(sigsqr, roots, ma, np.atleast_1d(time), measerr_scale=scale, mu=mu)
        return qm + mu, qv

    def kalman_filter(self, bestfit="map"):
        """One-step predictive mean/variance at the data times (assess_fit's ingredients, carma_pack.py:687-744)."""
        idx = self.best_index() if bestfit == "map" else int(bestfit)
        sigsqr, roots, ma, mu, scale = self._params_at(idx)
        mean, var = self._series.filter(sigsqr, roots, ma, measerr_scale=scale, mu=mu)
        return mean + mu, var

    def simulate(self, time, bestfit="map", seed=None, npaths=1):
        """Conditional simulation of the light curve at `time` given the data (carma_pack.py:830-854 ->
        KalmanFilterp::Simulate): one device call for all times and all `npaths` paths (extension: the reference
        draws one path).  Returns an array of len(time), or (npaths, len(time)) for npaths > 1."""
        idx = self.best_index() if bestfit == "map" else int(bestfit)
        sigsqr, roots, ma, mu, scale = self._params_at(idx)
        if seed is None:
            seed = int(np.random.SeedSequence().generate_state(1, dtype=np.uint64)[0] >> 1)
        out = self._series.simulate(sigsqr, roots, ma, np.atleast_1d(time), measerr_scale=scale, mu=mu, seed=seed, npaths=npaths)
        return out[0] if npaths == 1 else out

    def psd_credible_band(self, percentile=68.0, nsamples=None, freq=None, seed=0):
        """Numeric part of plot_power_spectrum (carma_pack.py:548-612): pointwise credibility band of the
        power spectrum over the posterior.  Returns (psd_lo, psd_hi, psd_mid, freq)."""
        sigmas = np.ravel(self._samples["sigma"])
        ar_coefs = self._samples["ar_coefs"]
        ma_coefs = self._samples["ma_coefs"]
        n = sigmas.size
        if nsamples is None or nsamples > n:
            nsamples = n
        pick = np.random.default_rng(seed).permutation(n)[:nsamples]
        if freq is None:
            dt = np.diff(self.time)
            freq = np.logspace(np.log10(1.0 / (self.time.max() - self.time.min())), np.log10(0.5 / dt.min()), 200)
        s = 2.0j * np.pi * freq
        num = np.zeros((nsamples, freq.size), dtype=complex)
        den = np.zeros((nsamples, freq.size), dtype=complex)
        for k in range(ma_coefs.shape[1]):
            num += ma_coefs[pick, k:k + 1] * s[None, :] ** k
        for k in range(ar_coefs.shape[1]):
            den += ar_coefs[pick, k:k + 1] * s[None, :] ** (ar_coefs.shape[1] - 1 - k)
        psd = sigmas[pick, None] ** 2 * np.abs(num) ** 2 / np.abs(den) ** 2
        lo, hi = (100.0 - percentile) / 2.0, 100.0 - (100.0 - percentile) / 2.0
        return np.percentile(psd, lo, axis=0), np.percentile(psd, hi, axis=0), np.median(psd, axis=0), freq

    def assess_fit_values(self, bestfit="map", nlags=20):
        """Numeric part of assess_fit (carma_pack.py:687-744): standardized one-step residuals and the
        autocorrelation of the residuals and of their squares (white under a good fit)."""
        mean, var = self.kalman_filter(bestfit)
        resid = (self.y - mean) / np.sqrt(var)

        def acf(x):
            x = x - x.mean()
            full = np.correlate(x, x, mode="full")[x.size - 1:]
            return full[:nlags + 1] / full[0]

        return resid, acf(resid), acf(resid ** 2), 1.96 / np.sqrt(resid.size)

    def DIC(self):  # carma_pack.py:808-828
        loglik = np.ravel(self._samples["loglik"])
        return -2.0 * loglik.mean() + 2.0 * np.var(-2.0 * loglik) / 2.0


class Car1Sample(MCMCSample):
    """MCMC samples of a CAR(1) model (carma_pack.py:866-1035, values only)."""

    def __init__(self, time, y, ysig, sampler=None, filename=None, trace=None, logpost=None, series=None, prior=None):
        """Reference signature (carma_pack.py:870): Car1Sample(time, y, ysig, sampler, filename=None)."""
        if sampler is not None:
            trace = np.array([list(r) for r in sampler.getSamples()], dtype=float)
            logpost = np.array(list(sampler.GetLogLikes()), dtype=float)
        if trace is None or logpost is None:
            raise ValueError("Car1Sample needs either a sampler object or trace and logpost arrays")
        trace = np.asarray(trace, dtype=float)
        logpost = np.asarray(logpost, dtype=float)
        super(Car1Sample, self).__init__(trace=trace, logpost=logpost)
        time, y, ysig = np.asarray(time, float), np.asarray(y, float), np.asarray(ysig, float)
        self.time, self.y, self.ysig = time, y, ysig
        self.p, self.q = 1, 0
        self._series_obj = series
        self._prior_obj = prior
        self._samples["var"] = trace[:, 0] ** 2
        self._samples["measerr_scale"] = trace[:, 1]
        self._samples["mu"] = trace[:, 2]
        self._samples["log_omega"] = trace[:, 3]
        omega = np.exp(trace[:, 3])
        self._samples["sigma"] = np.sqrt(2.0 * omega * trace[:, 0] ** 2)
        # the reference's per-sample getLogDensity loop (carma_pack.py:902-905) returns the stored log-posterior again
        self._samples["loglik"] = logpost.copy()
        self._samples["loglik_only"] = logpost - CarmaSample.log_prior(trace)
        self._trace = trace
        self.parameters = list(self._samples.keys())
        self.newaxis()

    @property
    def _series(self):
        if self._series_obj is None:
            self._series_obj = Series(self.time, self.y, self.ysig)
        return self._series_obj

    @property
    def _prior(self):
        if self._prior_obj is None:
            self._prior_obj = self._series.default_prior(True)
        return self._prior_obj

    def recompute_loglik(self):
        return self._series.loglik(KIND_CAR1, 1, 0, self._trace, prior=self._prior)
