"""Adaptive tempered Sequential Monte Carlo: posterior draws and the model evidence from full launches.

N particles move from the prior to the posterior through the tempered targets prior x L^beta, beta
going from 0 to 1.  Each stage picks the next beta so that the effective sample size (ESS) of the
incremental weights L^(beta' - beta) is ess_target * N, adds log mean(incremental weights) to log Z,
resamples systematically and then moves every particle with n_moves random-walk Metropolis sweeps
at beta'.  A sweep evaluates the proposals of all particles in ONE likelihood launch (N x n_meas
independent trajectories), so the sampler runs in the GPU's throughput regime, unlike a tempering
chain whose iteration is as slow as its slowest trajectory.

Several GPUs: each rank evaluates its comm.shard(n) block of every launch and the log-likelihoods
are all-gathered; every decision is then taken on every rank from the same generator, so the result
does not depend on the number of ranks.
"""
from __future__ import annotations

import os
import secrets
from time import perf_counter

import numpy as np

from .laplace import load_irf_tables
from .max_likelihood import _FAILED, _sigma
from .parallel import Comm
from .sim_utils import History, Ensemble
from .trial_move_generation import _approve_rows

MAX_PRIOR_DRAWS = 1000          # rejection draws per particle before the prior's support counts as empty
TARGET_ACCEPT = 0.234           # random-walk Metropolis acceptance rate the scale lambda is steered to


def prior_box(ensemble_fields):
    """(lo, hi) of the active parameters in the sampler's coordinates: log10 of the prior_dist bounds
    where do_log is set, the bounds themselves otherwise.  The box must be finite and not empty, with a
    positive lower bound for log parameters."""
    ef = ensemble_fields
    lo, hi = [], []
    for i in np.flatnonzero(ef["active"]):
        name = ef["names"][i]
        a, b = (float(v) for v in ef["prior_dist"][name])
        if not (np.isfinite(a) and np.isfinite(b) and a < b) or (ef["do_log"][i] and a <= 0):
            raise ValueError(f"smc needs a finite, non-empty prior box with a positive lower bound for "
                             f"log parameters; {name} has {(a, b)}")
        lo.append(np.log10(a) if ef["do_log"][i] else a)
        hi.append(np.log10(b) if ef["do_log"][i] else b)
    return np.array(lo), np.array(hi)


def make_cuda_loglik(ensemble_fields, sigma, device=None, kernel="warp"):
    """The likelihood smc() uses on the GPU: states [n, n_params] -> log L [n] at temperature 1, summed
    over the measurements, one launch (eval_trial_moves).  A NaN, and any curve that failed (status
    bits), gives -inf."""
    from .trial_move_evaluation import PathCache, eval_trial_moves
    cache = PathCache(ensemble_fields, device=device, kernel=kernel)

    def loglik(states):
        res = eval_trial_moves(states, np.ones(len(states)), sigma, ensemble_fields, cache=cache)
        return np.where(np.any((res.status & _FAILED) != 0, axis=1), -np.inf, res.logll)
    return loglik


def _ess(logw):
    """(ESS, max, sum of exp(logw - max)) of unnormalised log weights."""
    m = np.max(logw)
    w = np.exp(logw - m)
    s = w.sum()
    return s * s / np.dot(w, w), m, s


def _incremental(dbeta, ll):
    """log of L^dbeta for dbeta > 0, with L = 0 (ll = -inf) kept at -inf."""
    return np.where(np.isneginf(ll), -np.inf, dbeta * ll)


def next_beta(beta, ll, target):
    """The beta' in (beta, 1] at which the ESS of the weights L^(beta' - beta) is `target`, by
    bisection; 1 if the ESS at 1 is at least `target`.  When no step reaches it (fewer particles with
    L > 0 than `target`), the smallest step the bisection resolves."""
    if _ess(_incremental(1.0 - beta, ll))[0] >= target:
        return 1.0
    lo, hi = 0.0, 1.0 - beta
    while True:
        mid = 0.5 * (lo + hi)
        if mid <= lo or mid >= hi:
            break
        if _ess(_incremental(mid, ll))[0] >= target:
            lo = mid
        else:
            hi = mid
    return beta + (lo if lo > 0 else hi)


def systematic_resample(rng, w):
    """N indices drawn systematically (one uniform) from the non-negative weights w [N]."""
    n = len(w)
    cdf = np.cumsum(w)
    pos = (rng.random() + np.arange(n)) * (cdf[-1] / n)
    return np.minimum(np.searchsorted(cdf, pos, side="right"), np.flatnonzero(w > 0)[-1])


def _root(cov):
    """A square root L (L L^T = cov) of a symmetric positive semi-definite matrix."""
    ev, V = np.linalg.eigh(0.5 * (cov + cov.T))
    return V * np.sqrt(np.maximum(ev, 0.0))


def smc(sim_info, iniPar, e_data, MCMC_fields, param_info, n_particles=4096, ess_target=0.5,
        n_moves=5, seed=None, export_path=None, comm=None, kernel="warp", irf_dir="IRFs",
        evaluator_factory=None, logger=None):
    """Adaptive tempered SMC on the problem metro() would sample; returns an Ensemble of the particles.

    Same config dicts as metro() (copied, not consumed).  The prior is uniform on the prior_dist box of
    the active parameters in the sampler's coordinates (log10 where do_log is set, linear otherwise),
    restricted by the checks trial_move_generation._approve_rows makes (p0 > n0, tauN and tauP within
    two decades): the target metro() samples under hard_bounds.  That prior is used whatever
    hard_bounds says.  The evidence log Z is relative to it, normalised over its support, so it
    depends on the box.  Inactive parameters stay at init_guess.  The likelihood is that of a _T == 1
    chain (its model uncertainty) at temperature 1; tempering multiplies log L by beta.

    n_particles >= 2; ess_target in (0, 1): the ESS each reweighting keeps, as a share of N; n_moves
    Metropolis sweeps per stage with the Gaussian proposal (2.38^2 / d) lambda Sigma, Sigma the
    weighted particle covariance of the active coordinates and lambda steered by the previous sweep's
    acceptance rate.  A proposal outside the prior's support is rejected without being simulated.
    After beta reaches 1, one more stage of sweeps.  All randomness comes from
    np.random.default_rng(seed), consumed the same way on every rank (seed None: rank 0 picks one).

    comm: a parallel.Comm; each rank evaluates its block of every launch.  kernel: as for PathCache.
    evaluator_factory(ensemble_fields) -> loglik(states [n, n_params]) -> [n] replaces the CUDA
    likelihood (tests); NaN counts as -inf either way.

    The result has one chain per particle, all at _T = 1, with latest_iter = 1: H.states[:, :, 0] are
    the final equal-weight particles and H.loglikelihood[:, 0] their log L, so
    posterior_predictive(result, burn_in=0) applies.  MS_list.smc holds log_evidence, seed,
    prior_draws and per-stage arrays beta, ess, acceptance (mean over the stage's sweeps), lam (the
    lambda of its last sweep), launches, trajectories and wall_time (s); stage 0 is the draw from the
    prior.  export_path: pickled into output_path as mle() does (rank 0).
    """
    clock0 = perf_counter()
    comm = comm or Comm()
    n_particles = int(n_particles)
    if n_particles < 2:
        raise ValueError("n_particles must be at least 2")
    if not 0 < ess_target < 1:
        raise ValueError("ess_target must lie in (0, 1)")
    if int(n_moves) != n_moves or n_moves < 1:
        raise ValueError("n_moves must be a positive integer")
    MCMC_fields = dict(MCMC_fields)
    MCMC_fields.setdefault("num_iters", 1)
    MCMC_fields.setdefault("checkpoint_freq", 1)
    MS_list = Ensemble(dict(param_info), sim_info, MCMC_fields, 1)
    ef = MS_list.ensemble_fields
    if ef.get("do_mu_constraint", None) is not None:
        raise ValueError("smc does not sample under do_mu_constraint")
    if not ef["log_y"]:
        raise NotImplementedError("the likelihood kernel compares log10 signals (log_y = 1)")
    lo, hi = prior_box(ef)
    cold = [uf for uf in MS_list.unique_fields if uf["_T"] == 1]
    if not cold:
        raise ValueError("no chain at temperature 1: the likelihood is that of a _T == 1 chain")
    uf = cold[0]
    sigma = _sigma(uf)
    ef["_init_params"] = iniPar
    ef["_times"], ef["_vals"], ef["_uncs"] = e_data
    if ef.get("irf_convolution", None) is not None:
        ef["_IRF_tables"] = load_irf_tables(ef["irf_convolution"], irf_dir)
    else:
        ef["_IRF_tables"] = None
    if evaluator_factory is not None:
        loglik = evaluator_factory(ef)
    else:
        loglik = make_cuda_loglik(ef, sigma, device=comm.local_rank, kernel=kernel)
    if seed is None:
        seed = int(comm.broadcast_array(np.array([secrets.randbits(52)], dtype=np.float64))[0])
    rng = np.random.default_rng(seed)

    N = n_particles
    n_meas = int(ef["_sim_info"]["num_meas"])
    active = np.asarray(ef["active"], dtype=bool)
    do_log = np.asarray(ef["do_log"], dtype=bool)
    d = int(active.sum())
    log_cols, lin_cols = np.flatnonzero(active & do_log), np.flatnonzero(active & ~do_log)
    base = MS_list.H.states[0, :, 0].copy()
    with np.errstate(divide="ignore", invalid="ignore"):
        base_log = np.where(do_log, np.log10(base), base)

    def supported(x):
        full = np.repeat(base_log[None, :], len(x), axis=0)
        full[:, active] = x
        with np.errstate(over="ignore", invalid="ignore"):
            return _approve_rows(full, ef)

    def linear(x):
        states = np.repeat(base[None, :], len(x), axis=0)
        states[:, log_cols] = 10 ** x[:, do_log[active]]
        states[:, lin_cols] = x[:, ~do_log[active]]
        return states

    def evaluate(x):
        """log L of the sampler-coordinate points x [n, d]: one launch, this rank's block."""
        n = len(x)
        r0, r1 = comm.shard(n)
        local = np.asarray(loglik(linear(x[r0:r1])), dtype=np.float64) if r1 > r0 else np.zeros(0)
        ll = comm.allgather_rows(local[:, None], n)[:, 0]
        return np.where(np.isnan(ll), -np.inf, ll)

    rec = {k: [] for k in ("beta", "ess", "acceptance", "lam", "launches", "trajectories", "wall_time")}

    def record(beta, ess, acc, lam, launches, traj, t0):
        for k, v in zip(rec, (beta, ess, acc, lam, launches, traj, perf_counter() - t0)):
            rec[k].append(v)
        if logger is not None:
            logger.info(f"SMC stage {len(rec['beta']) - 1}: beta {beta:.6g} ESS {ess:.1f} acceptance {acc:.3f} "
                        f"lambda {lam:.3g} launches {launches} log Z {log_z:.6f}")

    # stage 0: the prior, by rejection from the box
    t0 = perf_counter()
    x = np.empty((N, d))
    got = draws = 0
    while got < N:
        if draws >= MAX_PRIOR_DRAWS * N:
            raise ValueError(f"the prior's support is (nearly) empty: {got} of {draws} draws from the box "
                             "passed the checks (p0 > n0, tauN and tauP within two decades)")
        cand = rng.uniform(lo, hi, size=(N, d))
        draws += N
        ok = cand[supported(cand)][:N - got]
        x[got:got + len(ok)] = ok
        got += len(ok)
    ll = evaluate(x)
    log_z = 0.0
    lam = 1.0
    record(0.0, float(N), np.nan, lam, 1, N * n_meas, t0)
    if not np.any(np.isfinite(ll)):
        raise ValueError("no particle drawn from the prior has a finite likelihood")

    beta = 0.0
    final = False
    while True:
        t0 = perf_counter()
        if beta < 1.0:
            new_beta = next_beta(beta, ll, ess_target * N)
            if not new_beta > beta:
                raise RuntimeError(f"tempering cannot advance from beta = {beta!r}: the particles' log-likelihoods "
                                   "spread too far for a step that double precision resolves")
            logw = _incremental(new_beta - beta, ll)
            ess, m, s = _ess(logw)
            log_z += m + np.log(s) - np.log(N)
            w = np.exp(logw - m)
            w /= w.sum()
            cov = np.atleast_2d(np.cov(x, rowvar=False, aweights=w))
            idx = systematic_resample(rng, w)
            x, ll = x[idx], ll[idx]
            beta = new_beta
        else:
            final = True
            ess = float(N)
            cov = np.atleast_2d(np.cov(x, rowvar=False))
        root = _root(cov * (2.38 ** 2 / d))
        launches = traj = 0
        acc_sum = 0.0
        for _ in range(int(n_moves)):
            z = rng.standard_normal((N, d))
            u = rng.random(N)
            prop = x + np.sqrt(lam) * (z @ root.T)
            inside = supported(prop)
            new_ll = np.full(N, -np.inf)
            if inside.any():
                new_ll[inside] = evaluate(prop[inside])
                launches += 1
                traj += int(inside.sum()) * n_meas
            with np.errstate(invalid="ignore", over="ignore"):
                accept = inside & (u < np.exp(beta * (new_ll - ll)))
            x[accept], ll[accept] = prop[accept], new_ll[accept]
            rate = float(accept.mean())
            acc_sum += rate
            lam_used = lam
            lam *= np.exp(2.0 * (rate - TARGET_ACCEPT))
        record(beta, float(ess), acc_sum / n_moves, lam_used, launches, traj, t0)
        if final:
            break

    H = History(N, 1, ef["names"])
    H.states[:, :, 0] = linear(x)
    H.loglikelihood[:, 0] = ll
    MS_list.H = H
    ef["_T"] = [1] * N
    ef["_n_chains"] = N
    ef["do_parallel_tempering"] = False
    uf = dict(uf, _T=1)
    MS_list.unique_fields = [uf] * N
    MS_list.latest_iter = 1
    MS_list.smc = {"log_evidence": float(log_z), "seed": seed, "prior_draws": draws,
                   **{k: np.array(v, dtype=np.int64 if k in ("launches", "trajectories") else float)
                      for k, v in rec.items()}}
    if logger is not None:
        logger.info(f"SMC: {len(rec['beta'])} stages, {int(np.sum(rec['launches']))} launches, "
                    f"log Z {log_z:.6f}, {perf_counter() - clock0:.3f} s")
    if export_path is not None and comm.rank == 0:
        os.makedirs(ef["output_path"], exist_ok=True)
        MS_list.checkpoint(os.path.join(ef["output_path"], export_path))
    return MS_list
