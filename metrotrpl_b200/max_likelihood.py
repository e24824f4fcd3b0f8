"""Maximum-likelihood driver, mirroring MLE/max_likelihood.py.

The reference minimises the negative log-likelihood of one state with SciPy's Nelder-Mead, one
forward simulation of every measurement per function call (max_likelihood.py:11-110, :148-150).
Nelder-Mead is sequential, but what it may ask for next is known in advance: the reflection, the
expansion and the two contractions of the current simplex (or, after a failed contraction, the
N shrunk vertices).  ``nelder_mead_batched`` evaluates those candidates in ONE batched likelihood
call per iteration and then takes exactly the decisions SciPy's ``_minimize_neldermead`` takes
(same coefficients, initial simplex, ordering and termination tests), so the iterates are SciPy's
as long as the function values are.  ``nelder_mead_multi`` runs K such searches side by side, one
call for the candidates of all of them, so that many starts fill a launch that one start leaves
nearly empty.  ``mle`` keeps the reference's signature and adds ``starts``;
``best_fit_covariance`` gives the Laplace approximation at the best fit.
"""
from __future__ import annotations

import os

import numpy as np

from .laplace import load_irf_tables
from .sim_utils import Ensemble

DEFAULT_NUM_ITERS = 1000        # max_likelihood.py:10


_MESSAGES = ("Optimization terminated successfully.",
             "Maximum number of function evaluations has been exceeded.",
             "Maximum number of iterations has been exceeded.")


def nelder_mead_multi(fun_batch, X0, xatol=1e-4, fatol=1e-4, maxiter=None, maxfev=None, callback=None):
    """K independent Nelder-Mead searches with SciPy's rules, started from the rows of X0[K, N].

    Each iteration makes one ``fun_batch(X[n, N]) -> f[n]`` call with the reflection, expansion and
    both contractions of every running simplex, and at most one more with the shrunk vertices of the
    simplices that shrink.  Every simplex takes the decisions, termination tests and counters SciPy's
    ``_minimize_neldermead`` takes from its start, including where the evaluation budget runs out in
    the middle of an iteration (the candidates SciPy could not afford are evaluated but not used); a
    simplex that has converged or hit a limit drops out of the batch.  As long as f of a point does
    not depend on which other points share its call, start k's result is SciPy's from X0[k].

    callback(idx, x[len(idx), N], f[len(idx)]) after every iteration: the simplices that took it and
    their best vertices.  Returns a dict of per-start arrays x [K, N], fun, nit, nfev, message (list),
    final_simplex (sim [K, N+1, N], fsim [K, N+1]), and the batched calls made (nbatch) and points
    evaluated (npoints) by the whole search.
    """
    rho, chi, psi, sigma = 1.0, 2.0, 0.5, 0.5
    X0 = np.atleast_2d(np.asarray(X0, dtype=float))
    K, N = X0.shape
    sim = np.repeat(X0[:, None, :], N + 1, axis=1)
    for k in range(N):                       # scipy: nonzdelt = 0.05, zdelt = 0.00025
        y = X0[:, k]
        sim[:, k + 1, k] = np.where(y != 0, (1 + 0.05) * y, 0.00025)
    if maxiter is None and maxfev is None:
        maxiter = maxfev = N * 200
    elif maxiter is None:
        maxiter = N * 200 if maxfev == np.inf else np.inf
    elif maxfev is None:
        maxfev = N * 200 if maxiter == np.inf else np.inf
    n0 = int(min(N + 1, maxfev))             # SciPy stops the initial evaluations at maxfev
    fsim = np.full((K, N + 1), np.inf)
    nbatch = npoints = 0
    if n0 > 0:
        fsim[:, :n0] = np.asarray(fun_batch(sim[:, :n0].reshape(-1, N)), dtype=float).reshape(K, n0)
        nbatch, npoints = 1, K * n0
    nfev = np.full(K, n0)
    nit = np.ones(K, dtype=int)
    for _ in range(2):                       # scipy sorts twice before its loop
        ind = np.argsort(fsim, axis=1)
        sim, fsim = np.take_along_axis(sim, ind[:, :, None], 1), np.take_along_axis(fsim, ind, 1)
    converged = np.zeros(K, dtype=bool)
    while True:
        run = np.flatnonzero(~converged & (nfev < maxfev) & (nit < maxiter))
        S, F = sim[run], fsim[run]
        conv = ((np.abs(S[:, 1:] - S[:, :1]).max(axis=(1, 2), initial=0.0) <= xatol)
                & (np.abs(F[:, :1] - F[:, 1:]).max(axis=1, initial=0.0) <= fatol))
        converged[run[conv]] = True
        run, S, F = run[~conv], S[~conv], F[~conv]
        if run.size == 0:
            break
        R = len(run)
        xbar = S[:, 0].copy()                # np.add.reduce(sim[:-1], 0): row after row
        for j in range(1, N):
            xbar += S[:, j]
        xbar /= N
        worst = S[:, -1]
        cand = np.stack([(1 + rho) * xbar - rho * worst,
                         (1 + rho * chi) * xbar - rho * chi * worst,
                         (1 + psi * rho) * xbar - psi * rho * worst,
                         (1 - psi) * xbar + psi * worst], axis=1)
        fc = np.asarray(fun_batch(cand.reshape(-1, N)), dtype=float).reshape(R, 4)
        nbatch += 1
        npoints += 4 * R
        fxr, fxe, fxc, fxcc = fc.T
        budget = maxfev - nfev[run] - 1      # evaluations left after the reflection
        nfev[run] += 1
        c_e = fxr < F[:, 0]
        c_r = ~c_e & (fxr < F[:, -2])
        c_c = ~c_e & ~c_r & (fxr < F[:, -1])
        c_cc = ~c_e & ~c_r & ~c_c
        second = c_e | c_c | c_cc            # cases that evaluate a second point
        paid = ~second | (budget >= 1)
        nfev[run[second & paid]] += 1
        budget = budget - second
        pick = np.select([c_e & (fxe < fxr), c_e | c_r, c_c & (fxc <= fxr), c_cc & (fxcc < F[:, -1])],
                         [1, 0, 2, 3], -1)
        shrink = paid & (pick < 0)
        move = paid & (pick >= 0)
        rows = np.flatnonzero(move)
        S[rows, -1] = cand[rows, pick[rows]]
        F[rows, -1] = fc[rows, pick[rows]]
        complete = paid.copy()
        if shrink.any():
            rows = np.flatnonzero(shrink)
            b = budget[rows]
            j = np.arange(N)[None, :]
            shrunk = j < np.minimum(N, b + 1)[:, None]       # vertices 1..N moved before SciPy's call fails
            paid_v = j < np.minimum(N, b)[:, None]           # and those it could evaluate
            Sh = S[rows]
            Sh[:, 1:] = np.where(shrunk[:, :, None], Sh[:, :1] + sigma * (Sh[:, 1:] - Sh[:, :1]), Sh[:, 1:])
            Fh = F[rows]
            if paid_v.any():
                f1 = Fh[:, 1:]
                f1[paid_v] = np.asarray(fun_batch(Sh[:, 1:][paid_v]), dtype=float)
                Fh[:, 1:] = f1
                nbatch += 1
                npoints += int(paid_v.sum())
            S[rows], F[rows] = Sh, Fh
            nfev[run[rows]] += paid_v.sum(axis=1)
            complete[rows] = b >= N
        nit[run[complete]] += 1
        ind = np.argsort(F, axis=1)
        S, F = np.take_along_axis(S, ind[:, :, None], 1), np.take_along_axis(F, ind, 1)
        sim[run], fsim[run] = S, F
        if callback is not None:
            callback(run, S[:, 0].copy(), F[:, 0].copy())
    message = [_MESSAGES[1] if nfev[k] >= maxfev else _MESSAGES[2] if nit[k] >= maxiter else _MESSAGES[0]
               for k in range(K)]
    return {"x": sim[:, 0].copy(), "fun": np.min(fsim, axis=1), "nit": nit, "nfev": nfev, "message": message,
            "nbatch": nbatch, "npoints": npoints, "final_simplex": (sim, fsim)}


def _one_start(res, k):
    """Start k of a nelder_mead_multi result, with nelder_mead_batched's keys."""
    sim, fsim = res["final_simplex"]
    return {"x": res["x"][k], "fun": float(res["fun"][k]), "nit": int(res["nit"][k]), "nfev": int(res["nfev"][k]),
            "nbatch": res["nbatch"], "npoints": res["npoints"], "message": res["message"][k],
            "final_simplex": (sim[k], fsim[k])}


def nelder_mead_batched(fun_batch, x0, xatol=1e-4, fatol=1e-4, maxiter=None, maxfev=None, callback=None):
    """Nelder-Mead with SciPy's rules from one start: nelder_mead_multi with K = 1.

    Returns a dict with x, fun, nit, nfev (the evaluations SciPy would have made), nbatch (the
    batched calls actually made), npoints (points actually evaluated) and message.
    """
    cb = None if callback is None else (lambda idx, x, f: callback(x[0], f[0]))
    x0 = np.asarray(x0, dtype=float).ravel()
    return _one_start(nelder_mead_multi(fun_batch, x0[None, :], xatol, fatol, maxiter, maxfev, cb), 0)


def _sigma(fields):
    """The model uncertainty per measurement type the likelihood uses (max_likelihood.py:95)."""
    sigma = fields.get("current_sigma", None) or fields.get("model_uncertainty", None)
    if sigma is None:
        raise KeyError("current_sigma")            # max_likelihood.py:95 reads MCMC_fields["current_sigma"]
    return sigma


def draw_starts(ensemble_fields, state, n_starts, seed=None):
    """n_starts states: row 0 is `state`, rows 1.. draw every active parameter from its prior_dist box
    (log-uniform where do_log is set, uniform otherwise, column by column as dense_sampling.random_grid
    does) with np.random.default_rng(seed); inactive parameters keep their value in `state`."""
    ef = ensemble_fields
    n_starts = int(n_starts)
    if n_starts < 1:
        raise ValueError("starts must be at least 1")
    rng = np.random.default_rng(seed)
    out = np.repeat(np.asarray(state, dtype=float)[None, :], n_starts, axis=0)
    for i in np.flatnonzero(ef["active"]):
        name = ef["names"][i]
        lo, hi = (float(b) for b in ef["prior_dist"][name])
        if not (np.isfinite(lo) and np.isfinite(hi) and 0 <= lo <= hi) or (ef["do_log"][i] and lo == 0):
            raise ValueError(f"drawing starts needs a finite prior box with a positive lower bound for "
                             f"log-uniform parameters; {name} has {(lo, hi)}")
        if lo == hi:
            out[1:, i] = lo
        elif ef["do_log"][i]:
            out[1:, i] = 10 ** rng.uniform(np.log10(lo), np.log10(hi), n_starts - 1)
        else:
            out[1:, i] = rng.uniform(lo, hi, n_starts - 1)
    return out


def mle(e_data, sim_params, param_info, init_params, sim_flags, export_path, logger, evaluator=None,
        irf_dir="IRFs", device=None, kernel="warp", starts=None, seed=None):
    """Same call and result as max_likelihood.py:113-160: the Ensemble whose single chain holds the
    visited states (column k = k-th accepted best vertex) and their log-likelihoods.

    evaluator(states[n, n_params]) -> logll[n] may be injected (tests); by default the CUDA path.
    kernel="seulex": the low-latency integrator (PathCache) - a simplex iteration is a handful of
    trajectories, i.e. pure latency.

    starts: None searches from init_guess alone, as the reference does.  An int K searches from K
    starts at once (nelder_mead_multi: one launch holds the candidates of every running simplex):
    init_guess and K - 1 draws from prior_dist (draw_starts, seeded by `seed`).  An array
    [K, n_params] gives the starts; its active columns are used, inactive parameters stay at
    init_guess.  Every start walks SciPy's Nelder-Mead path from where it starts.  The Ensemble is
    that of the best start (lowest cost; the first on a tie): its chain begins at that start's state,
    and MS_list.opt describes it with the single-start keys (nbatch / npoints count the whole search)
    plus "best_start" and "starts", the per-start x0, x, fun, nit, nfev and message.
    """
    sigma = _sigma(sim_flags)
    sim_flags = dict(sim_flags)
    sim_flags.setdefault("num_iters", DEFAULT_NUM_ITERS)
    sim_flags.setdefault("checkpoint_freq", DEFAULT_NUM_ITERS)
    MS_list = Ensemble(param_info, sim_params, sim_flags, DEFAULT_NUM_ITERS)
    ef = MS_list.ensemble_fields
    ef["_init_params"] = init_params
    ef["_times"], ef["_vals"], ef["_uncs"] = e_data
    if ef.get("irf_convolution", None) is not None:
        ef["_IRF_tables"] = load_irf_tables(ef["irf_convolution"], irf_dir)
    else:
        ef["_IRF_tables"] = None
    if not ef["log_y"]:
        raise NotImplementedError("the likelihood kernel compares log10 signals (log_y = 1)")
    active = ef["active"]
    base = MS_list.H.states[0, :, 0].copy()
    if starts is None:
        start_states = base[None, :]
    elif np.ndim(starts) == 0:
        start_states = draw_starts(ef, base, starts, seed)
    else:
        start_states = np.array(starts, dtype=float, ndmin=2)
        if start_states.shape[1] != len(base) or len(start_states) < 1:
            raise ValueError(f"starts must be [K, {len(base)}] states, got {start_states.shape}")
        start_states[:, ~active] = base[~active]
    if not np.all(start_states[:, active] > 0):
        raise ValueError("the search runs in log10 of the active parameters: starts must be positive")
    if evaluator is None:
        from .trial_move_evaluation import PathCache, eval_trial_moves
        cache = PathCache(ef, device=device, kernel=kernel)

        def evaluator(states):
            return eval_trial_moves(states, np.ones(len(states)), sigma, ef, cache=cache).logll

    def cost_batch(X):
        states = np.repeat(base[None, :], len(X), axis=0)
        states[:, active] = 10 ** np.asarray(X)
        ll = np.asarray(evaluator(states), dtype=float)
        return np.where(np.isfinite(ll), -ll, np.inf)

    K = len(start_states)
    steps = []                                   # (simplices, best vertices, costs) per iteration
    best_cost = np.full(K, np.inf)

    def progress(idx, x, f):
        steps.append((idx, x, f))
        best_cost[idx] = f
        if logger is not None:
            if starts is None:
                logger.info(f"Iter {len(steps)} Cost: {f[0]}")
            else:
                logger.info(f"Iter {len(steps)} Running: {len(idx)} Cost: {np.min(best_cost)}")

    X0 = np.log10(start_states[:, active])
    res = nelder_mead_multi(cost_batch, X0, callback=progress)
    b = int(np.argmin(res["fun"]))
    opt = _one_start(res, b)

    H = MS_list.H
    H.states[0, :, 0] = start_states[b]
    MS_list.latest_iter = 1
    for idx, x, f in steps:
        i = np.searchsorted(idx, b)
        if i == len(idx) or idx[i] != b:
            continue
        k = MS_list.latest_iter
        if k >= H.accept.shape[1]:
            H.extend(2 * H.accept.shape[1])
        H.states[0, :, k] = H.states[0, :, k - 1]
        H.states[0, active, k] = 10 ** x[i]
        H.loglikelihood[0, k] = -f[i]
        MS_list.latest_iter = k + 1
    if logger is not None:
        if starts is not None:
            logger.info(f"Best of {K} starts: {b}")
        logger.info(10 ** opt["x"])
        logger.info(-opt["fun"])
        logger.info(opt["message"])
    MS_list.opt = {k: v for k, v in opt.items() if k != "final_simplex"}
    if starts is not None:
        MS_list.opt["best_start"] = b
        MS_list.opt["starts"] = {"x0": X0, "x": res["x"], "fun": res["fun"], "nit": res["nit"],
                                 "nfev": res["nfev"], "message": res["message"]}
    if MS_list.latest_iter < H.accept.shape[1]:
        H.truncate(MS_list.latest_iter)
    if export_path is not None:
        os.makedirs(ef["output_path"], exist_ok=True)
        MS_list.checkpoint(os.path.join(ef["output_path"], export_path))
    return MS_list


# status bits after which a curve says nothing about the parameters (the tail floored at DBL_MIN and
# the explicit-path marker are not failures)
_FAILED = 1 | 2 | 4 | 16 | 32 | 64      # MAX_STEPS, H_UNDERFLOW, NONFINITE, NEG_FRAC, NAN_LL, CONV_FAIL


def fits_by_measurement(prob, fit, status, per_meas):
    """Split the fitted curves of a run with TRPL_OPT_FIT by measurement: (fits, vals, uncs), where
    fits[m] is [n_sets, n_t] - NaN past the compared points, and everywhere for a set whose curve m
    failed (status bits or a non-finite log-likelihood) - and vals[m], uncs[m] are the data."""
    fits, vals, uncs = [], [], []
    for m in range(prob.n_meas):
        sl = slice(int(prob.t_off[m]), int(prob.t_off[m] + prob.n_t[m]))
        f = np.array(fit[:, sl], dtype=float)
        f[((status[:, m] & _FAILED) != 0) | ~np.isfinite(per_meas[:, m, 0])] = np.nan
        fits.append(f)
        vals.append(prob.vals[sl])
        uncs.append(prob.uncs[sl])
    return fits, vals, uncs


def best_fit_covariance(MS_list, step=1e-4, device=None, kernel="warp", evaluator=None):
    """Laplace approximation at the best state of an MLE chain (its last column), in the log10 scale
    of the active parameters that mle() searches in.

    One batch of 2P + 1 states - the best one and +-step in log10 of each active parameter - gives the
    Jacobian J_m of every fitted curve over its compared points by central differences, and the
    Gauss-Newton precision H = 2 sum_m sum_k J_mk J_mk^T / (sigma_m^2 + 2 u_k^2) of the reference's
    log-likelihood -sum (fit - vals)^2 / (sigma^2 + 2 u^2) (no 1/2 there, hence the 2).  cov = H^-1.

    evaluator(states[n, n_params]) -> (fits, vals, uncs, sigmas) may be injected (tests), with fits,
    vals and uncs per measurement as fits_by_measurement gives them and sigmas[m] the model
    uncertainty of measurement m; by default the CUDA path.

    Returns a dict: names, x (log10 best state), cov, std, corr, precision, grad (central-difference
    gradient of the log-likelihood: ~0 at an optimum), ok and reason.  ok is False and cov, std and
    corr are NaN when an evaluation failed, the compared points of a curve differ between the states,
    or H is not positive definite (a parameter the data do not identify).
    """
    ef = MS_list.ensemble_fields
    active = np.asarray(ef["active"], dtype=bool)
    names = [n for n, a in zip(ef["names"], active) if a]
    state = np.array(MS_list.H.states[0, :, -1], dtype=float)
    x = np.log10(state[active])
    P = len(x)
    X = np.repeat(x[None, :], 2 * P + 1, axis=0)
    for i in range(P):
        X[1 + 2 * i, i] += step
        X[2 + 2 * i, i] -= step
    states = np.repeat(state[None, :], 2 * P + 1, axis=0)
    states[1:, active] = 10 ** X[1:]
    if evaluator is None:
        from .trial_move_evaluation import PathCache, eval_trial_moves
        sigma = _sigma(MS_list.unique_fields[0])
        cache = PathCache(ef, device=device, kernel=kernel)

        def evaluator(states):
            res = eval_trial_moves(states, np.ones(len(states)), sigma, ef, cache=cache, want_fit=True)
            return (*fits_by_measurement(cache.prob, res.fit, res.status, res.per_meas),
                    [sigma[t] for t in ef["_sim_info"]["meas_types"]])

    fits, vals, uncs, sigmas = evaluator(states)
    nan = np.full((P, P), np.nan)
    out = {"names": names, "x": x, "cov": nan, "std": np.full(P, np.nan), "corr": nan.copy(),
           "precision": nan.copy(), "grad": np.full(P, np.nan), "ok": False, "reason": ""}
    prec = np.zeros((P, P))
    ll = np.zeros(2 * P + 1)
    for m, f in enumerate(fits):
        f = np.asarray(f, dtype=float)
        n_c = np.where(np.isnan(f).any(axis=1), np.argmax(np.isnan(f), axis=1), f.shape[1])
        bad = np.flatnonzero((n_c == 0) | ~np.isfinite(np.where(np.isnan(f), 0.0, f)).all(axis=1))
        if bad.size:
            out["reason"] = f"evaluation failed: measurement {m}, state {int(bad[0])} of the +-step batch"
            return out
        if np.any(n_c != n_c[0]):
            out["reason"] = f"compared points of measurement {m} change between the +-step states"
            return out
        n = n_c[0]
        w = 1.0 / (sigmas[m] ** 2 + 2 * np.asarray(uncs[m], dtype=float)[:n] ** 2)
        J = (f[1::2, :n] - f[2::2, :n]).T / (2 * step)         # [n, P]
        prec += 2 * (J.T * w) @ J
        ll -= ((f[:, :n] - np.asarray(vals[m], dtype=float)[:n]) ** 2 * w).sum(axis=1)
    out["precision"] = prec
    out["grad"] = (ll[1::2] - ll[2::2]) / (2 * step)
    ev = np.linalg.eigvalsh(prec)
    if not ev[0] > P * np.finfo(float).eps * ev[-1]:
        out["reason"] = "precision not positive definite: a parameter (or combination) the data do not identify"
        return out
    cov = np.linalg.inv(prec)
    cov = 0.5 * (cov + cov.T)
    std = np.sqrt(np.diag(cov))
    out.update(cov=cov, std=std, corr=cov / np.outer(std, std), ok=True)
    return out
