"""Host mirror of trial_move_evaluation.py: log-likelihood of proposed states, in batches.

``eval_trial_move`` keeps the reference's call (trial_move_evaluation.py:9-28) for one state.
``eval_trial_moves`` evaluates many states (one per chain, or a dense-sampling block) in one
launch; this is the form metropolis.py and dense_sampling.py use.

What runs where: the whole of one_sim_likelihood (trial_move_evaluation.py:30-166) - simulation,
trim, negative test, min_y floor, log10 residual, weighted sum - runs inside the CUDA kernel; the
host only packs parameters and reads back one scalar per (state, measurement, temperature).
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Optional, Sequence

import numpy as np

from . import _capi
from .forward_solver import get_context
from .utils import search_c_grps


@dataclass
class BatchLikelihood:
    """Result of one batched evaluation."""
    logll: np.ndarray        # [n_sets]            sum over measurements at each state's own temperature
    per_meas: np.ndarray     # [n_sets, n_meas, 3] per-curve log-likelihood at the three temperatures
    status: np.ndarray       # [n_sets, n_meas]
    nsteps: np.ndarray       # [n_sets, n_meas, 2]
    curves: Optional[np.ndarray] = None
    fit: Optional[np.ndarray] = None        # [n_sets, n_times_total] fitted curves (want_fit=True)
    problem: Optional[_capi.PackedProblem] = field(default=None, repr=False)   # for fitted()

    def at_temperature(self, slot: int) -> np.ndarray:
        """Sum over measurements at temperature slot 0..2 (the ll_funcs of the reference)."""
        return self.per_meas[:, :, slot].sum(axis=1)

    def fitted(self, m: int, s: int = 0):
        """(times, fit, vals, uncs) of measurement m for parameter set s, cut to the points the
        likelihood compared: fit - vals are its residuals, log10(model) - log10(data).  Without an IRF
        that is every point; with one, the times inside the convolved span.  Empty when the
        convolution failed.  Needs eval_trial_moves(..., want_fit=True)."""
        if self.fit is None:
            raise ValueError("no fitted curves: evaluate with want_fit=True")
        prob = self.problem
        sl = slice(int(prob.t_off[m]), int(prob.t_off[m] + prob.n_t[m]))
        f = self.fit[s, sl]
        done = np.flatnonzero(~np.isnan(f))
        n_c = int(done[-1]) + 1 if done.size else 0        # compared points are a prefix; NaN after it
        return prob.times[sl][:n_c], f[:n_c], prob.vals[sl][:n_c], prob.uncs[sl][:n_c]


class PathCache:
    """Packs shared_fields once and keeps the problem resident on the device."""

    def __init__(self, shared_fields, device=None, ctx=None, kernel="warp"):
        """ctx: a private _capi.Context (own stream and device buffers) instead of the process-wide
        one of `device`; two caches on two contexts let consecutive launches overlap.
        kernel: "warp" (RODAS4, one trajectory per warp: throughput), "cta" (RODAS4 on a whole CTA,
        csrc/cta_trajectory.h; 'std' model with nx = 128 only, refused at launch otherwise) or
        "seulex" (order-6 extrapolation, one trajectory per CTA, csrc/extrapolation.h: half the
        latency for batches of a few hundred trajectories - single states, Nelder-Mead simplices,
        tempering ladders; 'std' or 'traps' model with nx = 128 only)."""
        sf = shared_fields
        if any(m == "pa" for m in sf["_sim_info"]["meas_types"]):
            raise NotImplementedError("'pa' toy measurements are not simulations; not on the CUDA path")
        self.sf = sf
        self.prob = _capi.pack_problem(sf["_sim_info"], sf["_init_params"], sf["_times"], sf["_vals"],
                                       sf["_uncs"], model=sf.get("model", "std"),
                                       ini_mode=sf.get("ini_mode", "density"),
                                       irf_convolution=sf.get("irf_convolution", None),
                                       irf_tables=sf.get("_IRF_tables", None))
        self.ctx = ctx if ctx is not None else get_context(device)
        self.ctx.set_problem(self.prob)
        self.n_meas = self.prob.n_meas
        idx = sf["_param_indexes"]
        self.idx = idx

        def group_index(spec, tag):
            """per-measurement state index of the _f/_a/_s parameter, or -1 (lines 38-60)."""
            out = np.full(self.n_meas, -1, dtype=np.int64)
            if spec is None:
                return out
            for m in range(self.n_meas):
                if m in spec[1]:
                    if spec[2] is not None and len(spec[2]) > 0:
                        name = f"{tag}{search_c_grps(spec[2], m)}"
                    else:
                        name = f"{tag}{m}"
                    out[m] = idx[name]
            return out

        if sf.get("ini_mode", "density") != "fluence" and (sf.get("fittable_fluences", None) is not None
                                                             or sf.get("fittable_absps", None) is not None):
            # trial_move_evaluation.py:44,51 multiplies iniPar[0] / iniPar[1] whatever the mode; with a
            # density profile those are the first two nodes' densities, not a fluence or an absorption
            # coefficient.  That is not reproduced; it is refused.
            raise ValueError("fittable_fluences / fittable_absps need ini_mode == 'fluence'")
        self.f_idx = group_index(sf.get("fittable_fluences", None), "_f")
        self.a_idx = group_index(sf.get("fittable_absps", None), "_a")
        self.s_idx = group_index(sf.get("scale_factor", None), "_s")
        self.flags = _capi.OPT_FORCE_MIN_Y if sf.get("force_min_y", False) else 0
        if kernel == "seulex":
            _capi.check_extrapolation_problem(sf.get("model", "std"), sf["_sim_info"]["nx"])
            self.flags |= _capi.OPT_EXTRAPOLATION | _capi.OPT_CTA_PER_TRAJ
        elif kernel == "cta":
            self.flags |= _capi.OPT_CTA_PER_TRAJ
        elif kernel != "warp":
            raise ValueError(f"unknown kernel {kernel!r}")

    def opts(self, honor_hmax=False):
        sf = self.sf
        return _capi.make_opts(sf.get("rtol", None), sf.get("atol", None), hmax=sf.get("hmax", 0.0),
                               honor_hmax=honor_hmax, flags=self.flags)

    def pack(self, states, sigmas, temps):
        """states [n_sets, n_params]; sigmas: dict meas_type -> sigma or [n_sets] of dicts;
        temps [n_sets, 3]."""
        sf = self.sf
        states = np.atleast_2d(np.asarray(states, dtype=np.float64))
        n_sets = states.shape[0]
        params = _capi.pack_params(states, self.idx, sf["units"], model=sf.get("model", "std"))
        aux = np.zeros((n_sets, self.n_meas, _capi.NAUX))
        aux[..., _capi.A_FLUENCE_MULT] = 1.0
        aux[..., _capi.A_ABSORB_MULT] = 1.0
        for m in range(self.n_meas):
            if self.f_idx[m] >= 0:
                aux[:, m, _capi.A_FLUENCE_MULT] = states[:, self.f_idx[m]]
            if self.a_idx[m] >= 0:
                aux[:, m, _capi.A_ABSORB_MULT] = states[:, self.a_idx[m]]
            if self.s_idx[m] >= 0:
                aux[:, m, _capi.A_SCALE_SHIFT] = np.log10(states[:, self.s_idx[m]])
        mtypes = sf["_sim_info"]["meas_types"]
        if isinstance(sigmas, dict):
            sig = np.broadcast_to(np.array([sigmas[t] for t in mtypes], dtype=np.float64), (n_sets, self.n_meas))
        elif len(sigmas) > 0 and all(s is sigmas[0] for s in sigmas):
            sig = np.broadcast_to(np.array([sigmas[0][t] for t in mtypes], dtype=np.float64), (n_sets, self.n_meas))
        else:
            sig = np.array([[s[t] for t in mtypes] for s in sigmas], dtype=np.float64)
        temps = np.asarray(temps, dtype=np.float64).reshape(n_sets, 3)
        for k in range(3):
            aux[:, :, _capi.A_S2T0 + k] = sig ** 2 * temps[:, k][:, None]
        return params, aux


def eval_trial_moves(states, temps, sigmas, shared_fields, cache: Optional[PathCache] = None,
                     want_curves=False, honor_hmax=False, want_fit=False) -> BatchLikelihood:
    """Log-likelihood of many proposed states in one launch.

    temps : [n_sets] (own temperature) or [n_sets, 3] (own + two others, e.g. the swap partners').
    want_fit : also return the fitted curves, what the likelihood compared with the data point by
        point (BatchLikelihood.fit, BatchLikelihood.fitted); no other result changes.
    """
    if cache is None:
        cache = PathCache(shared_fields)
    states = np.atleast_2d(np.asarray(states, dtype=np.float64))
    n_sets = states.shape[0]
    temps = np.asarray(temps, dtype=np.float64)
    if temps.ndim == 1:
        temps = np.repeat(temps[:, None], 3, axis=1)
    params, aux = cache.pack(states, sigmas, temps)
    cache.ctx.set_problem_if_needed(cache.prob)
    opts = cache.opts(honor_hmax)
    if want_fit:
        opts.flags |= _capi.OPT_FIT
    per, status, nsteps, curves = cache.ctx.loglik_batch(params, aux, opts, want_curves=want_curves)
    fit = cache.ctx.download_fit() if want_fit else None
    logll = per[:, :, 0].sum(axis=1)
    logll = np.where(np.isnan(logll), -np.inf, logll)
    return BatchLikelihood(logll, per, status, nsteps, curves, fit, cache.prob if want_fit else None)


def eval_trial_move(state, unique_fields, shared_fields, logger=None, cache=None):
    """Single-state call with the reference's signature (trial_move_evaluation.py:9-28).

    Returns (logll, ll_funcs) where ll_funcs[i](T) re-evaluates measurement i's likelihood at
    temperature T.  The reference builds closures over err_sq arrays; here T must be one of the
    temperatures the kernel evaluated: the chain's own ``_T`` and ``unique_fields.get("_T_alt")``.
    """
    T = unique_fields.get("_T", 1)
    alts = list(unique_fields.get("_T_alt", ()))[:2]
    tlist = [T] + alts + [T] * (2 - len(alts))
    res = eval_trial_moves(np.asarray(state, dtype=np.float64)[None, :], np.array([tlist]),
                           unique_fields["model_uncertainty"], shared_fields, cache=cache)

    def make(i):
        table = {float(t): res.per_meas[0, i, k] for k, t in enumerate(tlist)}

        def ll_func(temp):
            try:
                return table[float(temp)]
            except KeyError:
                raise KeyError(f"temperature {temp} was not evaluated; pass it in unique_fields['_T_alt']")
        return ll_func

    return float(res.logll[0]), [make(i) for i in range(res.per_meas.shape[1])]
