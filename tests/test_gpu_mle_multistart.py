"""GPU tier: many-start maximum likelihood through CUDA, and the covariance of its best fit.

Every start of mle(starts=K) must equal SciPy's Nelder-Mead driven by the same CUDA likelihood one
point at a time, bit for bit, and a single-start mle() from that start: a per-trajectory result of
the library does not depend on which other trajectories share its launch, so the batched search is K
searches side by side."""
import copy
import os
import tempfile

import numpy as np
import pytest
from scipy.optimize import minimize

from metrotrpl_b200 import _capi
from metrotrpl_b200.max_likelihood import best_fit_covariance, draw_starts, fits_by_measurement, mle
from metrotrpl_b200.trial_move_evaluation import PathCache, eval_trial_moves

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
STD_REL_TOL = 1e-6          # std of the best fit, CUDA vs the host lock-step build at rtol 1e-9; measured 5.5e-10


def _inputs(g, names, sim_info, ini, e_data, model, ini_mode, sigma, active, guess, prior, tmp):
    """mle()'s positional arguments for a fixture: (e_data, sim_info, param_info, ini, MCMC)."""
    param_info = {"names": list(names), "active": {n: int(n in active) for n in names},
                  "unit_conversions": {n: float(u) for n, u in zip(names, g["units"])},
                  "do_log": {n: 1 for n in names}, "prior_dist": {n: (0, np.inf) for n in names},
                  "init_guess": dict({n: float(v) for n, v in zip(names, g["states"][0])}, **guess),
                  "trial_move": {n: 0.05 for n in names}}
    param_info["prior_dist"].update(prior)
    MCMC = {"init_cond_path": "x", "measurement_path": "y", "output_path": tmp, "num_iters": 10,
            "solver": ("solveivp",), "model": model, "ini_mode": ini_mode, "log_y": 1, "checkpoint_freq": 10,
            "rtol": 1e-7, "atol": None, "current_sigma": {"TRPL": sigma}}
    return e_data, sim_info, param_info, ini, MCMC


def staub_mle_inputs(tmp):
    """The six-curve staub problem (tests/golden/staub6.npz, 'std', nx = 128), fitting tauN and Sf
    from a start away from the state the data were made with."""
    g = np.load(os.path.join(GOLDEN, "staub6.npz"))
    names = [str(n) for n in g["names"]]
    sim = {"lengths": list(g["lengths"]), "nx": [int(g["nx"])] * 6, "meas_types": ["TRPL"] * 6, "num_meas": 6}
    e_data = ([g["t"]] * 6, list(g["vals"]), list(g["uncs"]))
    return _inputs(g, names, sim, g["ini"], e_data, "std", "density", float(g["sigma"]), ("Sf", "tauN"),
                   {"tauN": 1500.0, "Sf": 2.0}, {"tauN": (50.0, 5e3), "Sf": (0.1, 1e3)}, tmp)


def traps_mle_inputs(tmp):
    """The trap-assisted problem of tests/golden/traps_irf.npz on 128 nodes, without the IRF (the
    grid the extrapolation integrator serves), fitting tauN and Nt."""
    g = np.load(os.path.join(GOLDEN, "traps_irf.npz"))
    names = [str(n) for n in g["names"]]
    sim = {"lengths": list(g["lengths"]), "nx": [128] * 2, "meas_types": ["TRPL"] * 2, "num_meas": 2}
    e_data = ([g["t"]] * 2, list(g["vals"]), list(g["uncs"]))
    return _inputs(g, names, sim, g["inis"], e_data, "traps", "fluence", 1.0, ("tauN", "Nt"),
                   {"tauN": 150.0, "Nt": 1e16}, {"tauN": (20.0, 5e3), "Nt": (1e14, 1e17)}, tmp)


def cuda_cost(ms, kernel):
    """Cost of one log10 point through the CUDA likelihood, as mle() computes it."""
    ef = ms.ensemble_fields
    cache = PathCache(ef, kernel=kernel)
    sigma = ms.unique_fields[0]["current_sigma"]
    base = ms.H.states[0, :, 0].copy()
    act = ef["active"]

    def cost(x):
        st = base.copy()
        st[act] = 10 ** np.asarray(x)
        ll = eval_trial_moves(st[None, :], np.ones(1), sigma, ef, cache=cache).logll[0]
        return -ll if np.isfinite(ll) else np.inf
    return cost


def check_starts(make_inputs, n_starts, seed, kernel):
    tmp = tempfile.mkdtemp()
    ms = mle(*make_inputs(tmp), None, None, kernel=kernel, starts=n_starts, seed=seed)
    st = ms.opt["starts"]
    b = ms.opt["best_start"]
    assert ms.opt["fun"] == st["fun"][b] == st["fun"].min()
    # every start: SciPy's search on the same likelihood, one point per launch
    cost = cuda_cost(ms, kernel)
    for k in range(n_starts):
        ref = minimize(cost, st["x0"][k], method="Nelder-Mead")
        assert np.array_equal(st["x"][k], ref.x) and st["fun"][k] == ref.fun, k
        assert (st["nit"][k], st["nfev"][k], st["message"][k]) == (ref.nit, ref.nfev, ref.message), k
    # every start: a single-start mle() from its state
    e_data, sim_info, param_info, ini, MCMC = make_inputs(tmp)
    names = param_info["names"]
    base = np.array([param_info["init_guess"][n] for n in names], dtype=float)
    ef = ms.ensemble_fields
    states = draw_starts(ef, base, n_starts, seed)
    for k in range(n_starts):
        e_data, sim_info, param_info, ini, MCMC = make_inputs(tmp)
        param_info["init_guess"] = dict(zip(names, states[k]))
        one = mle(e_data, sim_info, param_info, ini, MCMC, None, None, kernel=kernel)
        assert np.array_equal(one.opt["x"], st["x"][k]) and one.opt["fun"] == st["fun"][k], k
        assert (one.opt["nit"], one.opt["nfev"]) == (st["nit"][k], st["nfev"][k]), k
        if k == b:
            np.testing.assert_array_equal(one.H.states, ms.H.states)
            np.testing.assert_array_equal(one.H.loglikelihood, ms.H.loglikelihood)
    print(f"{kernel}: {n_starts} starts, best {b}, cost {ms.opt['fun']:.9g} (start 0: {st['fun'][0]:.9g}), "
          f"nit {st['nit'].min()}..{st['nit'].max()}, {ms.opt['nbatch']} launches, {ms.opt['npoints']} points")
    return ms


@pytest.fixture(scope="module")
def staub_fit():
    return check_starts(staub_mle_inputs, 16, 7, "warp")


def test_many_starts_are_scipys_searches_warp(staub_fit):
    assert staub_fit.opt["message"].startswith("Optimization terminated")


def test_many_starts_are_scipys_searches_seulex_traps():
    check_starts(traps_mle_inputs, 8, 3, "seulex")


def test_covariance_cuda_vs_host_build(staub_fit):
    from tests.emu import emu
    ms = copy.deepcopy(staub_fit)
    ef = ms.ensemble_fields
    ef["rtol"] = 1e-9
    gpu = best_fit_covariance(ms)
    sigma = ms.unique_fields[0]["current_sigma"]["TRPL"]
    prob = _capi.pack_problem(ef["_sim_info"], ef["_init_params"], ef["_times"], ef["_vals"], ef["_uncs"])

    def host(states):
        params = _capi.pack_params(states, ef["_param_indexes"], ef["units"])
        aux = _capi.default_aux(len(states), prob.n_meas, [sigma] * prob.n_meas)
        ll, st, _, _, fit = emu.loglik_batch(prob, params, aux, _capi.make_opts(RTOL=1e-9), False, fit=True)
        return (*fits_by_measurement(prob, fit, st, ll), [sigma] * prob.n_meas)

    cpu = best_fit_covariance(ms, evaluator=host)
    assert gpu["ok"] and cpu["ok"], (gpu["reason"], cpu["reason"])
    rel = np.abs(gpu["std"] / cpu["std"] - 1)
    print(f"std {gpu['std']} (CUDA) vs {cpu['std']} (host): {rel.max():.2e}; grad {gpu['grad']}")
    assert rel.max() <= STD_REL_TOL
    np.testing.assert_allclose(gpu["corr"], cpu["corr"], atol=1e-6)
