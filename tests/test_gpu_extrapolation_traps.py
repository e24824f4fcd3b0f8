"""GPU tier: the trap-assisted model through the order-6 extrapolation integrator's kernels
(csrc/extrapolation.h) at nx = 128 - the cooperative kernel (six columns on the four warps of a CTA)
and its one-warp twin - and through the Python paths that select them: PathCache, metro, mle."""
import tempfile

import numpy as np
import pytest

from metrotrpl_b200 import _capi
from tests.emu import emu
from tests.test_extrapolation_traps import compare_with_truth, jittered_states, traps128_problem

pytestmark = pytest.mark.gpu

SEULEX_WARP = _capi.OPT_EXTRAPOLATION
SEULEX_CTA = _capi.OPT_EXTRAPOLATION | _capi.OPT_CTA_PER_TRAJ
LOGLL_FLOOR = -1e4


@pytest.fixture(scope="module")
def ctx():
    c = _capi.Context(0)
    yield c
    c.close()


def run(ctx, prob, params, aux, flags=0, **kw):
    ctx.set_problem(prob)
    return ctx.loglik_batch(params, aux, _capi.make_opts(RTOL=kw.pop("rtol", 1e-7), flags=flags, **kw),
                            want_curves=True)


def fixture_batch(n_jitter=0, seed=11):
    g, names, idx, prob = traps128_problem()
    states = g["states"] if n_jitter == 0 else np.concatenate([g["states"], jittered_states(g, names, n_jitter, seed)])
    params = _capi.pack_params(states, idx, g["units"], model="traps")
    return g, prob, params, _capi.default_aux(len(params), 2, [1.0] * 2)


def test_cooperative_traps_kernel_against_the_converged_truth(ctx):
    """Cooperative kernel, traps + IRF at nx = 128, rtol 1e-7, against RODAS4 at rtol 1e-10: the
    bounds of the host lock-step case (test_extrapolation_traps.py)."""
    g, prob, params, aux = fixture_batch()
    seulex = run(ctx, prob, params, aux, SEULEX_CTA)
    rodas = run(ctx, prob, params, aux)
    truth = run(ctx, prob, params, aux, rtol=1e-10)
    curve, ll, ratio = compare_with_truth(seulex, truth, rodas, len(g["t"]))
    print("curve", curve, "logll", ll, "step ratio", ratio)
    assert curve <= 5e-6
    assert ll <= 1e-6
    assert ratio < 0.5
    assert not np.any(seulex[1] & 7)


def test_two_integrators_agree_on_1024_jittered_traps_states(ctx):
    """configs[3]'s states on 128 nodes: 1024 sets jittered +-0.1 decade x 2 curves through RODAS4 (one
    warp per trajectory) and the cooperative extrapolation kernel.  Every curve point within twelve
    decades of its start agrees to 1e-4, every set's log-likelihood above -1e4 to 2e-6, no failure
    status, and the extrapolation integrator takes fewer than 0.45x RODAS4's steps.  Measured on the
    B200: 2.6e-6, 1.0e-6 (all 1024 sets above the floor), 0.404x (67.7 against 167.6 steps)."""
    g, names, idx, prob = traps128_problem()
    n = 1024
    params = _capi.pack_params(jittered_states(g, names, n, seed=20261020), idx, g["units"], model="traps")
    aux = _capi.default_aux(n, 2, [1.0] * 2)
    ll_r, st_r, ns_r, cur_r = run(ctx, prob, params, aux)
    ll_x, st_x, ns_x, cur_x = run(ctx, prob, params, aux, SEULEX_CTA)
    nt = len(g["t"])
    R, X = cur_r.reshape(n, 2, nt), cur_x.reshape(n, 2, nt)
    in_range = R >= 1e-12 * R[:, :, :1]
    with np.errstate(all="ignore"):
        e = np.where(in_range, np.abs(X / R - 1), 0.0)
    tot_r, tot_x = ll_r[:, :, 0].sum(axis=1), ll_x[:, :, 0].sum(axis=1)
    ok = tot_r > LOGLL_FLOOR
    rel = np.abs(tot_x[ok] / tot_r[ok] - 1)
    ratio = ns_x[..., 0].mean() / ns_r[..., 0].mean()
    print("max curve difference", e.max(), "sets above the floor", int(ok.sum()), "max logll difference",
          rel.max(), "mean steps", ns_r[..., 0].mean(), ns_x[..., 0].mean(), "ratio", ratio)
    assert e.max() <= 1e-4
    assert ok.sum() > 100
    assert rel.max() <= 2e-6
    assert np.all((st_x & 7) == 0) and np.all((st_r & 7) == 0)
    assert ratio < 0.45


def test_one_warp_and_cooperative_traps_kernels_agree_bit_for_bit(ctx):
    """The cooperative kernel exchanges (N, Q, T) of every column increment and combines them in the
    one-warp driver's order: same curves, log-likelihoods, status and step counts, in any queue
    order."""
    g, prob, params, aux = fixture_batch(n_jitter=124)
    ll_w, st_w, ns_w, cur_w = run(ctx, prob, params, aux, SEULEX_WARP)
    ll_c, st_c, ns_c, cur_c = run(ctx, prob, params, aux, SEULEX_CTA)
    np.testing.assert_array_equal(ns_c, ns_w)
    np.testing.assert_array_equal(cur_c, cur_w)
    np.testing.assert_array_equal(ll_c, ll_w)
    np.testing.assert_array_equal(st_c, st_w)
    ctx.set_queue_order(np.random.default_rng(2).permutation(params.shape[0] * 2))
    try:
        ll_p, st_p, ns_p, cur_p = run(ctx, prob, params, aux, SEULEX_CTA)
    finally:
        ctx.set_queue_order(None)
    np.testing.assert_array_equal(cur_p, cur_c)
    np.testing.assert_array_equal(ll_p, ll_c)
    np.testing.assert_array_equal(ns_p, ns_c)
    np.testing.assert_array_equal(st_p, st_c)


def test_cooperative_traps_kernel_matches_host_lockstep_build(ctx):
    """Same source, two compilers (nvcc contracts into FMAs, the host build does not): curves to
    5e-7, step counts within 5."""
    g, prob, params, aux = fixture_batch()
    o = _capi.make_opts(RTOL=1e-7, flags=SEULEX_WARP)
    ll_g, st_g, ns_g, cur_g = run(ctx, prob, params, aux, SEULEX_CTA)
    ll_e, st_e, ns_e, cur_e = emu.loglik_batch(prob, params, aux, o, True)
    np.testing.assert_allclose(cur_g, cur_e, rtol=5e-7)
    np.testing.assert_allclose(ll_g, ll_e, rtol=1e-6)
    assert np.abs(ns_g[..., 0] - ns_e[..., 0]).max() <= 5


def test_cooperative_traps_kernel_ladder_and_min_y_floor(ctx):
    """The tempering ladder through the cooperative traps kernel equals the three temperature slots of
    a plain call, its per-chain rows are their sums over the curves; force_min_y is the host lock-step
    build's to rounding."""
    g, prob, params, aux0 = fixture_batch(n_jitter=12)
    n = params.shape[0]
    aux = _capi.default_aux(n, 2, [1.0] * 2, temps=(1.0, 2.0, 8.0))
    ll, _, _, _ = run(ctx, prob, params, aux, SEULEX_CTA)
    ctx.set_ladder(np.array([1.0, 2.0, 8.0, 64.0]))
    aux1 = _capi.default_aux(n, 2, [1.0] * 2, temps=(1.0, 1.0, 1.0))
    ctx.loglik_batch(params, aux1, _capi.make_opts(RTOL=1e-7, flags=SEULEX_CTA | _capi.OPT_LADDER), want_curves=False)
    lad = ctx.download_ladder(n)
    np.testing.assert_allclose(lad[:, :, :3], ll, rtol=1e-12)
    assert np.all(lad[:, :, 3] > lad[:, :, 2])
    rows, _ = ctx.download_ladder_sums(n)
    np.testing.assert_allclose(rows, lad.sum(axis=1), rtol=1e-14)
    flags = SEULEX_CTA | _capi.OPT_FORCE_MIN_Y
    ll_f, st_f, _, _ = run(ctx, prob, params, aux, flags)
    ll_e, _, _, _ = emu.loglik_batch(prob, params, aux, _capi.make_opts(RTOL=1e-7, flags=flags), True)
    np.testing.assert_allclose(ll_f, ll_e, rtol=1e-6)
    assert not np.any(st_f & 7)


def test_step_log_flush_in_the_cooperative_traps_kernel(ctx):
    """A 0.06 ns step cap forces about 1700 steps per curve: the 1024-entry step log is flushed
    mid-run by warp 0 of the CTA.  Same curves and log-likelihoods as the uncapped run."""
    g, prob, params, aux = fixture_batch()
    params, aux = params[:2], aux[:2]
    free = run(ctx, prob, params, aux, SEULEX_CTA)
    capped = run(ctx, prob, params, aux, SEULEX_CTA, hmax=0.06, honor_hmax=True)
    print("steps free", free[2][..., 0].tolist(), "capped", capped[2][..., 0].tolist())
    assert capped[2][..., 0].min() > 1024 and free[2][..., 0].max() < 1024
    T = free[3]
    in_range = T >= 1e-12 * T.max()
    np.testing.assert_allclose(np.where(in_range, capped[3], 1.0), np.where(in_range, T, 1.0), rtol=3e-5)
    np.testing.assert_allclose(capped[0], free[0], rtol=2e-6)
    assert not np.any(capped[1] & 7)


def test_extrapolation_refuses_grids_other_than_128_nodes(ctx):
    """Traps or std at nx != 128 with the extrapolation flag: refused by the C ABI (both kernels) and
    by PathCache."""
    from metrotrpl_b200.trial_move_evaluation import PathCache
    g, names, idx, _ = traps128_problem()
    sim = {"lengths": list(g["lengths"]), "nx": [100] * 2, "meas_types": ["TRPL"] * 2, "num_meas": 2}
    prob = _capi.pack_problem(sim, g["inis"], [g["t"]] * 2, None, None, model="traps", ini_mode="fluence")
    params = _capi.pack_params(g["states"][:1], idx, g["units"], model="traps")
    std = _capi.pack_problem(dict(sim, nx=[64] * 2), g["inis"], [g["t"]] * 2, None, None, model="std",
                             ini_mode="fluence")
    for p in (prob, std):
        ctx.set_problem(p)
        for flags in (SEULEX_WARP, SEULEX_CTA):
            with pytest.raises(_capi.TrplError, match="nx = 128"):
                ctx.loglik_batch(params, _capi.default_aux(1, 2, [1.0] * 2),
                                 _capi.make_opts(flags=flags | _capi.OPT_NO_LIKELIHOOD), want_curves=True)
    sf = dict(_traps_shared_fields(), _sim_info=dict(sim, nx=[256] * 2))
    with pytest.raises(ValueError, match="nx = 128"):
        PathCache(sf, kernel="seulex")


# ---- the Python paths: metro and mle on a traps problem ---------------------------------------

ACTIVE = ("p0", "tauN", "tauP", "kC", "Nt")


def _traps_shared_fields():
    """shared_fields of a two-curve traps problem at nx = 128 (fluence mode, no IRF) whose data are
    the fixture's first state's curves, log10, with fixed noise."""
    from metrotrpl_b200.trial_move_evaluation import eval_trial_moves
    g, names, idx, _ = traps128_problem(irf=False)
    t = g["t"]
    sim = {"lengths": list(g["lengths"]), "nx": [128] * 2, "meas_types": ["TRPL"] * 2, "num_meas": 2}
    sf = {"_sim_info": sim, "_init_params": [i.copy() for i in g["inis"]], "_times": [t, t],
          "_vals": [np.zeros_like(t)] * 2, "_uncs": [np.full(len(t), 0.02)] * 2, "_param_indexes": idx,
          "units": g["units"], "model": "traps", "ini_mode": "fluence", "rtol": 1e-7, "atol": None}
    cur = eval_trial_moves(g["states"][:1], np.ones(1), {"TRPL": 1.0}, sf, want_curves=True).curves
    noise = np.random.default_rng(4).normal(0.0, 0.01, size=(2, len(t)))
    sf["_vals"] = [np.log10(cur[0, m * len(t):(m + 1) * len(t)]) + noise[m] for m in range(2)]
    return sf


def _metro_args(tmp, n_chains, num_iters):
    g, names, idx, _ = traps128_problem(irf=False)
    sf = _traps_shared_fields()
    param_info = {"names": names, "active": {n: int(n in ACTIVE) for n in names},
                  "unit_conversions": {n: float(u) for n, u in zip(names, g["units"])},
                  "do_log": {n: 1 for n in names}, "prior_dist": {n: (0, np.inf) for n in names},
                  "init_guess": {n: float(v) for n, v in zip(names, g["states"][0])},
                  "trial_move": {n: 0.05 for n in names}}
    MCMC = {"init_cond_path": "x", "measurement_path": "y", "output_path": tmp, "num_iters": num_iters,
            "solver": ("solveivp",), "model": "traps", "ini_mode": "fluence", "log_y": 1,
            "checkpoint_freq": num_iters, "hard_bounds": 1, "rtol": 1e-7, "atol": None,
            "model_uncertainty": {"TRPL": 0.05},
            "parallel_tempering": list(1.5 ** np.arange(n_chains)), "temper_freq": 2}
    return sf["_sim_info"], sf["_init_params"], (sf["_times"], sf["_vals"], sf["_uncs"]), MCMC, param_info


def test_metro_tempering_on_a_traps_problem_through_the_low_latency_kernel():
    """metro(kernel="seulex"): 16 replicas x 2 curves, swaps every second iteration.  It completes, swaps
    happen, and every chain's final log-likelihood equals a RODAS4 evaluation of its final state at its
    temperature to 2e-6 (measured 1.7e-6, on log-likelihoods of -0.09 to -25)."""
    from metrotrpl_b200.metropolis import metro
    from metrotrpl_b200.trial_move_evaluation import PathCache, eval_trial_moves
    with tempfile.TemporaryDirectory() as tmp:
        ms = metro(*_metro_args(tmp, 16, 12), export_path="traps.pik", install_signal_handlers=False,
                   kernel="seulex")
    ef = ms.ensemble_fields
    assert ms.H.swap_attempts.sum() > 0
    assert ms.H.accept[:, 1:].sum() > 0
    final = ms.H.states[:, :, -1]
    T = np.asarray(ef["_T"], dtype=float)
    ref = eval_trial_moves(final, T, {"TRPL": 0.05}, ef, cache=PathCache(ef)).logll
    got = ms.H.loglikelihood[:, -1]
    print("accepted", int(ms.H.accept[:, 1:].sum()), "swaps", int(ms.H.swap_accept.sum()),
          "max logll difference", np.abs(got / ref - 1).max())
    assert np.all(np.isfinite(got))
    np.testing.assert_allclose(got, ref, rtol=2e-6)


def test_mle_on_a_traps_problem_through_the_low_latency_kernel():
    """mle(kernel="seulex") from a perturbed start reaches the optimum mle(kernel="warp") reaches, within
    the Nelder-Mead tolerances: 1e-3 in log10 of the parameters (ten times xatol: the simplex stops
    anywhere inside xatol of its best vertex) and fatol = 1e-4 in the cost, plus the integrators' 2e-6
    relative agreement.  Measured: the same vertex, costs 8e-6 apart."""
    from metrotrpl_b200.max_likelihood import mle
    out = {}
    for kernel in ("warp", "seulex"):
        with tempfile.TemporaryDirectory() as tmp:
            sim_info, ini, e_data, MCMC, param_info = _metro_args(tmp, 1, 1)
            MCMC.pop("parallel_tempering")
            MCMC["current_sigma"] = {"TRPL": 0.05}
            for n in param_info["active"]:
                param_info["active"][n] = int(n in ("tauN", "kC"))
            param_info["init_guess"] = dict(param_info["init_guess"], tauN=700.0, kC=0.6e-7)
            ms = mle(e_data, sim_info, param_info, ini, MCMC, None, None, kernel=kernel)
        out[kernel] = ms.opt
        print(kernel, ms.opt["x"], ms.opt["fun"], ms.opt["nit"], ms.opt["message"])
    w, s = out["warp"], out["seulex"]
    assert s["message"].startswith("Optimization terminated")
    assert np.max(np.abs(s["x"] - w["x"])) <= 1e-3
    assert abs(s["fun"] - w["fun"]) <= 1e-4 + 2e-6 * abs(w["fun"])
