"""GPU tier: fitted curves (TRPL_OPT_FIT, trpl_download_fit) from every kernel family.

For each family: the fitted values equal the oracle's restatement of the reference's steps applied to
the kernel's own raw curves, they reproduce the log-likelihoods of the same run, and asking for them
changes no other output (tests/test_fit_curves.py holds the checks)."""
import numpy as np
import pytest

from metrotrpl_b200 import _capi
from metrotrpl_b200.trial_move_evaluation import eval_trial_moves
from tests import parity_cases as pc
from tests.emu import emu
from tests.test_fit_curves import (assert_no_side_effects, check_fit, conv_refused_case, staub_case,
                                   traps_irf_case)
from tests.test_extrapolation_traps import traps128_problem
from tests.test_gpu_parity import SLOW_DECAY_STATES

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    c = _capi.Context(0)
    yield c
    c.close()


def gpu_run(ctx, prob, params, aux, flags, rtol=1e-7):
    """(logll, status, nsteps, curves, fit) with TRPL_OPT_FIT, and (logll, status, nsteps, curves)
    of the same run without it."""
    ctx.set_problem(prob)
    opts = _capi.make_opts(RTOL=rtol, flags=flags | _capi.OPT_FIT)
    res = ctx.loglik_batch(params, aux, opts, want_curves=True)
    fit = ctx.download_fit()
    plain = ctx.loglik_batch(params, aux, _capi.make_opts(RTOL=rtol, flags=flags), want_curves=True)
    return (*res, fit), plain


def check_family(ctx, prob, params, aux, flags, tables=None, force_min_y=False):
    with_fit, without = gpu_run(ctx, prob, params, aux, flags)
    assert_no_side_effects(with_fit, without)
    ll, st, ns, cur, fit = with_fit
    n, n_short = check_fit(prob, aux, ll, st, cur, fit, irf_tables=tables, force_min_y=force_min_y)
    return with_fit, n, n_short


def fluence_std_case(nx):
    """'std' model on nx nodes, fluence mode (two curves, stiff and non-stiff states)."""
    names, units, idx = pc._known_units()
    guess = dict(pc.BASE, n0=1e8, p0=3e15, mu_n=20, mu_p=20, ks=4.8e-11, Cn=4.4e-29, Cp=4.4e-29,
                 Sf=10, Sb=1e3, tauN=511, tauP=871)
    st = np.array([[guess[n] for n in names], [dict(guess, tauN=40, tauP=60)[n] for n in names]], dtype=float)
    t = np.linspace(0, 50, 101)
    sim = {"lengths": [500.0, 311.0], "nx": [nx, nx], "meas_types": ["TRPL", "TRTS"], "num_meas": 2}
    inis = [np.array([2e12, 6e4, 1.0]), np.array([2e12, 6e4, -1.0])]
    prob = _capi.pack_problem(sim, inis, [t, t], [np.full(101, 16.0), np.full(101, -3.0)],
                              [np.full(101, 0.05)] * 2, ini_mode="fluence")
    aux = _capi.default_aux(2, 2, [1.0, 2.0], temps=(1.0, 4.0, 16.0))
    aux[:, 0, _capi.A_SCALE_SHIFT] = 0.3
    return prob, _capi.pack_params(st, idx, units), aux


@pytest.mark.parametrize("nx", [128, 100, 40])
def test_fit_warp_kernel_std(ctx, nx):
    """trpl_forward_kernel: padding-free (nx = 128, the staub fixture) and padded grids."""
    if nx == 128:
        prob, params, aux = staub_case()
    else:
        prob, params, aux = fluence_std_case(nx)
    check_family(ctx, prob, params, aux, 0)


def test_fit_explicit_path(ctx):
    """Non-stiff trajectories go to trpl_explicit_kernel; their fitted curves come the same way."""
    names, units, idx = pc._known_units()
    t = np.linspace(0, 100, 1001)
    sim = {"lengths": [2000, 2000], "nx": [128, 128], "meas_types": ["TRPL", "TRTS"], "num_meas": 2}
    ini = np.array([1e15 * np.ones(128), 3e15 * np.exp(-np.arange(128) / 40.0)])
    guess = dict(pc.BASE, n0=1e8, p0=1e17, ks=1e-13, tauN=4, tauP=6, Cn=1e-29, Cp=1e-29)
    stiff = dict(guess, mu_n=20, mu_p=20, Sf=10, Sb=10)
    st = np.array([[guess[n] for n in names], [stiff[n] for n in names]], dtype=float)
    prob = _capi.pack_problem(sim, ini, [t, t], [np.full(1001, 20.0), np.full(1001, -2.0)], [np.full(1001, 0.1)] * 2)
    aux = _capi.default_aux(2, 2, [1.0, 1.0])
    (ll, s, ns, cur, fit), n, _ = check_family(ctx, prob, _capi.pack_params(st, idx, units), aux, 0)
    assert np.all(s[0] & _capi.ST_EXPLICIT) and not np.any(s[1] & _capi.ST_EXPLICIT)


@pytest.mark.parametrize("nx", [256, 400])
def test_fit_team_kernels_traps_irf(ctx, nx):
    """Two-warp (nx = 256) and four-warp (nx = 400) teams, traps + IRF: the post pass."""
    prob, params, aux, tables = traps_irf_case(nx=nx)
    _, n, n_short = check_family(ctx, prob, params, aux, 0, tables)
    assert n_short == n


@pytest.mark.parametrize("flags", [_capi.OPT_EXTRAPOLATION, _capi.OPT_EXTRAPOLATION | _capi.OPT_CTA_PER_TRAJ],
                         ids=["seulex_warp", "seulex_cta"])
def test_fit_extrapolation_kernels_traps128_irf(ctx, flags):
    g, names, idx, prob = traps128_problem()
    params = _capi.pack_params(g["states"][:4], idx, g["units"], model="traps")
    aux = _capi.default_aux(4, 2, [1.0] * 2)
    aux[:, 0, _capi.A_SCALE_SHIFT] = 0.25
    check_family(ctx, prob, params, aux, flags, [(g["moments"], g["t_irf"])] * 2)


def test_fit_cta_kernel(ctx):
    prob, params, aux = staub_case()
    check_family(ctx, prob, params, aux, _capi.OPT_CTA_PER_TRAJ)


def test_fit_force_min_y_and_refused_convolution(ctx):
    prob, params, aux = staub_case(shift=-1.5)
    check_family(ctx, prob, params, aux, _capi.OPT_FORCE_MIN_Y, force_min_y=True)
    prob, params, aux, tables = conv_refused_case()
    (ll, st, ns, cur, fit), _, _ = check_family(ctx, prob, params, aux, 0, tables)
    assert np.all(st[:, 1] & _capi.ST_CONV_FAIL) and np.all(np.isnan(fit[:, prob.t_off[1]:]))


def test_fit_with_ladder_and_queue_order(ctx):
    """TRPL_OPT_LADDER (post pass with residual scratch) and an explicit queue order: the ladder rows
    and every other output unchanged by the fit."""
    prob, params, aux = staub_case(n=6)
    temps = np.array([1.0, 1.7, 3.1, 9.0])
    ctx.set_problem(prob)
    ctx.set_ladder(temps)
    aux = aux.copy()
    aux[..., _capi.A_S2T1] = aux[..., _capi.A_S2T0]          # sigma^2 at temperature 1
    (ll, st, ns, cur, fit), _, _ = check_family(ctx, prob, params, aux, _capi.OPT_LADDER)
    lad_plain = ctx.download_ladder(params.shape[0])
    ctx.loglik_batch(params, aux, _capi.make_opts(RTOL=1e-7, flags=_capi.OPT_LADDER | _capi.OPT_FIT), want_curves=True)
    np.testing.assert_array_equal(ctx.download_ladder(params.shape[0]), lad_plain)
    np.testing.assert_array_equal(ctx.download_fit(), fit)
    # explicit queue order: same fit, bit for bit
    n_traj = params.shape[0] * prob.n_meas
    ctx.set_queue_order(np.random.default_rng(2).permutation(n_traj))
    try:
        with_fit, without = gpu_run(ctx, prob, params, aux, 0)
    finally:
        ctx.set_queue_order(None)
    assert_no_side_effects(with_fit, without)
    ll0, st0, ns0, cur0, fit0 = gpu_run(ctx, prob, params, aux, 0)[0]
    np.testing.assert_array_equal(with_fit[4], fit0)


def test_fit_matches_host_lockstep_build(ctx):
    """Device fit equals the host build's to the tolerance of test_gpu_matches_host_lockstep_build, on
    the same states (curves that stay well above rounding noise)."""
    g, prob, params, aux = pc.staub_problem()
    sel = SLOW_DECAY_STATES[:4]
    for prob, params, aux in ((prob, params[sel], aux[sel]), traps_irf_case(nx=256, n=2)[:3]):
        (ll, st, ns, cur, fit), _ = gpu_run(ctx, prob, params, aux, 0)
        fit_e = emu.loglik_batch(prob, params, aux, _capi.make_opts(RTOL=1e-7), fit=True)[4]
        np.testing.assert_array_equal(np.isnan(fit), np.isnan(fit_e))
        ok = ~np.isnan(fit)
        np.testing.assert_allclose(fit[ok], fit_e[ok], rtol=5e-7)


def test_fit_refusals(ctx):
    prob, params, aux = staub_case(n=1)
    ctx.set_problem(prob)
    with pytest.raises(_capi.TrplError, match="TRPL_OPT_NO_LIKELIHOOD"):
        ctx.loglik_batch(params, aux, _capi.make_opts(flags=_capi.OPT_FIT | _capi.OPT_NO_LIKELIHOOD))
    ctx.loglik_batch(params, aux, _capi.make_opts())
    with pytest.raises(_capi.TrplError, match="did not produce fitted curves"):
        ctx.download_fit()
    g = np.load(pc.os.path.join(pc.GOLDEN, "staub6.npz"))
    sim = {"lengths": list(g["lengths"]), "nx": [int(g["nx"])] * 6, "meas_types": ["TRPL"] * 6, "num_meas": 6}
    ctx.set_problem(_capi.pack_problem(sim, g["ini"], [g["t"]] * 6))         # no vals / uncs
    with pytest.raises(_capi.TrplError, match="TRPL_OPT_FIT needs measurement values"):
        ctx.loglik_batch(params, aux, _capi.make_opts(flags=_capi.OPT_FIT))


def test_eval_trial_moves_fitted_round_trip():
    """eval_trial_moves(want_fit=True).fitted(m): the compared points of measurement m, whose
    residuals give back the per-curve log-likelihood."""
    g, names, idx, prob = traps128_problem()
    sf = {"_sim_info": {"lengths": list(g["lengths"]), "nx": [128] * 2, "meas_types": ["TRPL"] * 2, "num_meas": 2},
          "_init_params": g["inis"], "_times": [g["t"]] * 2, "_vals": list(g["vals"]), "_uncs": list(g["uncs"]),
          "_param_indexes": idx, "units": g["units"], "model": "traps", "ini_mode": "fluence", "rtol": 1e-7,
          "irf_convolution": [520, 520], "_IRF_tables": {520: (g["moments"], g["t_irf"])}}
    states = g["states"][:2]
    res = eval_trial_moves(states, np.array([1.0, 2.0]), {"TRPL": 1.0}, sf, want_fit=True)
    plain = eval_trial_moves(states, np.array([1.0, 2.0]), {"TRPL": 1.0}, sf)
    np.testing.assert_array_equal(res.per_meas, plain.per_meas)
    assert plain.fit is None and res.fit.shape == (2, 2 * len(g["t"]))
    for s, T in ((0, 1.0), (1, 2.0)):
        for m in range(2):
            t, f, v, u = res.fitted(m, s)
            assert 0 < len(t) < len(g["t"]) and np.all(np.isfinite(f))
            np.testing.assert_array_equal(t, g["t"][:len(t)])
            np.testing.assert_array_equal(v, g["vals"][m][:len(t)])
            want = -np.sum((f - v) ** 2 / (T + 2 * u ** 2))
            assert abs(want - res.per_meas[s, m, 0]) <= 1e-12 * abs(want)
