"""Posterior predictive bands: per-point quantiles of the fitted curves over the draws of a metro() run.

The figure of a Bayesian TRPL fit is the measured curve drawn over the band of model curves the
posterior allows.  ``posterior_predictive`` evaluates the posterior draws in one launch with fitted
curves (TRPL_OPT_FIT), and the quantiles of every compared point are selected on the device
(trpl_fit_quantiles): only [n_q][n_times_total] quantiles and the counts leave the GPU, never the
[n_draws][n_times_total] fitted values.
"""
from __future__ import annotations

import math

import numpy as np

from . import _capi
from .max_likelihood import _FAILED, _sigma


def select_draws(MS_list, burn_in=0.5, thin=1, max_draws=None, seed=None):
    """(chains, iters) of the posterior draws of an Ensemble: every chain whose unique_fields _T is 1,
    iterations k in [ceil(burn_in * latest_iter), latest_iter) with step thin, chain by chain.  With
    max_draws, a subset of that many drawn with np.random.default_rng(seed) without replacement, kept
    in the same order (so the result does not depend on the order of the draw)."""
    if not (0 <= burn_in < 1):
        raise ValueError("burn_in must lie in [0, 1)")
    if int(thin) != thin or thin < 1:
        raise ValueError("thin must be a positive integer")
    if max_draws is not None and (int(max_draws) != max_draws or max_draws < 1):
        raise ValueError("max_draws must be a positive integer or None")
    cold = [c for c, uf in enumerate(MS_list.unique_fields) if uf.get("_T", 1) == 1]
    if not cold:
        raise ValueError("no chain at temperature 1: the posterior draws come from the _T == 1 chains")
    n_iter = int(MS_list.latest_iter)
    iters = np.arange(math.ceil(burn_in * n_iter), n_iter, int(thin))
    chains = np.repeat(np.array(cold, dtype=np.int64), iters.size)
    iters = np.tile(iters, len(cold))
    if chains.size == 0:
        raise ValueError(f"no draws: latest_iter {n_iter} with burn_in {burn_in}")
    if max_draws is not None and chains.size > max_draws:
        keep = np.sort(np.random.default_rng(seed).choice(chains.size, int(max_draws), replace=False))
        chains, iters = chains[keep], iters[keep]
    return chains, iters


def posterior_predictive(MS_list, quantiles=(0.025, 0.5, 0.975), burn_in=0.5, thin=1, max_draws=None,
                         seed=None, device=None, kernel="warp", evaluator=None):
    """Posterior predictive band of every measurement of a metro() Ensemble.

    The draws are the states MS_list.H.states[c, :, k] of every chain c with _T == 1 (select_draws:
    burn_in, thin, and a seeded subset of max_draws).  All of them are evaluated in ONE launch with
    fitted curves, with the model uncertainty of a _T == 1 chain's unique_fields, and the quantiles of
    each point over the draws are taken on the device: np.nanquantile(fit, quantiles, axis=0,
    method="linear") bit for bit, where fit holds what the likelihood compared with the data (log10 of
    the signal plus the scale shift; NaN past the compared points of an IRF curve).  The fit of a draw
    whose evaluation failed enters as the kernel produced it; n_failed counts those draws.

    quantiles: 1 to 8 levels in [0, 1], ascending; the band is [first, last].  kernel: as for
    PathCache.  evaluator(states[n, n_params]) -> (quant [n_q, n_times_total], count [n_times_total],
    status [n, n_meas]) may be injected (tests); by default the CUDA path.

    One GPU only: exact quantiles of draws sharded over several GPUs would need all their fitted
    values in one place, which is what this routine avoids.

    Returns a dict: quantiles (the levels), n_draws, n_failed, chains and iters (the draws) and
    measurements, one dict per measurement with times, vals and uncs cut to the points any draw
    compared (count > 0), quantiles [n_q, n_c], count [n_c], and coverage, the share of those data
    points inside the band (NaN when there are none).
    """
    q = np.array(quantiles, dtype=np.float64, ndmin=1)
    if q.ndim != 1 or not 1 <= q.size <= _capi.MAX_QUANTILES:
        raise ValueError(f"quantiles: 1 to {_capi.MAX_QUANTILES} levels")
    if not np.all((q >= 0) & (q <= 1)):
        raise ValueError("quantiles must lie in [0, 1]")
    if np.any(np.diff(q) < 0):
        raise ValueError("quantiles must be ascending: the band is [quantiles[0], quantiles[-1]]")
    chains, iters = select_draws(MS_list, burn_in, thin, max_draws, seed)
    states = np.ascontiguousarray(MS_list.H.states[chains, :, iters], dtype=np.float64)
    ef = MS_list.ensemble_fields
    if evaluator is None:
        from .trial_move_evaluation import PathCache
        sigma = _sigma(MS_list.unique_fields[int(chains[0])])
        cache = PathCache(ef, device=device, kernel=kernel)

        def evaluator(states):
            params, aux = cache.pack(states, sigma, np.ones((len(states), 3)))
            cache.ctx.set_problem_if_needed(cache.prob)
            opts = cache.opts()
            opts.flags |= _capi.OPT_FIT
            _, status, _, _ = cache.ctx.loglik_batch(params, aux, opts)
            return (*cache.ctx.fit_quantiles(q), status)

    quant, count, status = evaluator(states)
    quant, count, status = np.asarray(quant), np.asarray(count), np.asarray(status)
    meas = []
    off = 0
    for m in range(int(ef["_sim_info"]["num_meas"])):
        t = np.asarray(ef["_times"][m], dtype=np.float64)
        sl = slice(off, off + t.size)
        off += t.size
        seen = count[sl] > 0
        v = np.asarray(ef["_vals"][m], dtype=np.float64)[seen]
        band = quant[:, sl][:, seen]
        inside = (v >= band[0]) & (v <= band[-1])
        meas.append({"times": t[seen], "vals": v, "uncs": np.asarray(ef["_uncs"][m], dtype=np.float64)[seen],
                     "quantiles": band, "count": count[sl][seen],
                     "coverage": float(inside.mean()) if v.size else float("nan")})
    return {"quantiles": q, "n_draws": int(len(states)),
            "n_failed": int(np.count_nonzero(np.any((status & _FAILED) != 0, axis=1))),
            "chains": chains, "iters": iters, "measurements": meas}
