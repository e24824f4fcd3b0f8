"""CPU tier: fitted curves (TRPL_OPT_FIT) in the host lock-step build of the kernel source.

The fitted curve of a trajectory is, point by point, what the likelihood compared with the data:
log10(|y|) + scale_shift after the min_y floor and, with an IRF, after convolution, max-shift and
trim; NaN past the compared points.  Checked here against the oracle's restatement of the
reference's steps applied to the build's own raw curves (exact to rounding) and against the
log-likelihoods the same run returned.  The host build runs the fit pass on the stored curves after
the run (emu.loglik_batch(..., fit=True)), as the library does, so it cannot change the run; the GPU
tier (test_gpu_fit_curves.py, which shares these helpers) checks that no output of the library
changes."""
import numpy as np

from metrotrpl_b200 import _capi
from oracle import trpl_oracle as orc
from tests import parity_cases as pc
from tests.emu import emu
from tests.test_extrapolation_traps import traps128_problem

# fitted values vs the oracle's steps on the same raw curve: 1e-14 absolute, or two units in the last
# place of the value (the device's log10 is not correctly rounded: 1 ulp is 1.4e-14 at |fit| ~ 100)
FIT_ABS_TOL = 1e-14
LOGLL_REL_TOL = 1e-12     # -sum (fit - vals)^2 / (sigma^2 T + 2 u^2) vs the run's own log-likelihoods


def oracle_fit(curve, t, vals, shift, irf_table=None, force_min_y=False):
    """The reference's err_sq left operand (trial_move_evaluation.py:117-166) on one raw curve, through
    the oracle: convolution with max-shift and trim, sign flip, set_min_y, log10 + shift.  NaN past
    the compared points, all NaN when the convolution fails."""
    out = np.full(len(t), np.nan)
    sol = np.array(curve, dtype=float)
    vv = np.asarray(vals, dtype=float)
    if irf_table is not None:
        try:
            ct, cy, ok = orc.irf_convolve(np.asarray(t, dtype=float), sol, irf_table, time_max_shift=True)
            if not ok:
                return out
            sol, _, vv, _ = orc.trim_after_convolution(ct, cy, np.asarray(t, dtype=float), vv, vv)
        except (ValueError, IndexError):
            return out
    sol = np.abs(sol)
    if force_min_y:
        sol, _, _ = orc.raise_to_min_y(sol, vv, shift)
    with np.errstate(divide="ignore"):
        out[:len(sol)] = np.log10(sol) + shift
    return out


def check_fit(prob, aux, ll, status, curves, fit, irf_tables=None, force_min_y=False):
    """Tests 1 and 2 for one run: fit against the oracle's steps on the run's own curves, and the
    run's log-likelihoods from fit.  irf_tables: per measurement (moments, t_irf) or None.
    Returns (number of trajectories checked, number with compared prefix shorter than n_t)."""
    n_sets = aux.shape[0]
    n_short = 0
    for s in range(n_sets):
        for m in range(prob.n_meas):
            sl = slice(int(prob.t_off[m]), int(prob.t_off[m] + prob.n_t[m]))
            t, v, u = prob.times[sl], prob.vals[sl], prob.uncs[sl]
            shift = aux[s, m, _capi.A_SCALE_SHIFT]
            want = oracle_fit(curves[s, sl], t, v, shift, None if irf_tables is None else irf_tables[m],
                              force_min_y)
            got = fit[s, sl]
            np.testing.assert_array_equal(np.isnan(got), np.isnan(want), err_msg=f"NaN pattern, set {s} meas {m}")
            ok = ~np.isnan(want)
            tol = np.maximum(FIT_ABS_TOL, 2 * np.spacing(np.abs(want[ok])))
            assert np.all(np.abs(got[ok] - want[ok]) <= tol), (s, m, np.abs(got[ok] - want[ok]).max())
            n_c = int(ok.sum())
            assert np.all(ok[:n_c]), "compared points are a prefix"
            n_short += n_c < len(t)
            if n_c == 0:
                assert status[s, m] & _capi.ST_CONV_FAIL and np.all(ll[s, m] == -np.inf)
                continue
            if not np.all(np.isfinite(ll[s, m])):
                continue
            r2 = (got[:n_c] - v[:n_c]) ** 2
            for k in range(3):
                want_ll = -np.sum(r2 / (aux[s, m, _capi.A_S2T0 + k] + 2 * u[:n_c] ** 2))
                assert abs(want_ll - ll[s, m, k]) <= LOGLL_REL_TOL * abs(ll[s, m, k]), (s, m, k, want_ll, ll[s, m, k])
    return n_sets * prob.n_meas, n_short


def assert_no_side_effects(with_fit, without_fit):
    """Test 3: logll, status, nsteps and curves bit-identical with and without the fit."""
    for a, b, name in zip(with_fit[:4], without_fit[:4], ("logll", "status", "nsteps", "curves")):
        np.testing.assert_array_equal(a, b, err_msg=name)


def emu_run(prob, params, aux, flags, rtol=1e-7):
    """(logll, status, nsteps, curves, fit) of the host build."""
    return emu.loglik_batch(prob, params, aux, _capi.make_opts(RTOL=rtol, flags=flags), fit=True)


def staub_case(n=4, shift=0.37):
    g, prob, params, aux = pc.staub_problem()
    aux = aux[:n].copy()
    aux[..., _capi.A_SCALE_SHIFT] = shift
    return prob, params[:n], aux


def traps_irf_case(nx=256, n=3, times=None):
    """configs[3]: traps + IRF on nx nodes (fluence mode: the initial condition follows the grid)."""
    g = np.load(pc.os.path.join(pc.GOLDEN, "traps_irf.npz"))
    names = [str(x) for x in g["names"]]
    idx = {x: i for i, x in enumerate(names)}
    t0 = g["t"]
    t = t0 if times is None else times
    vals = [np.interp(t, t0, g["vals"][m]) for m in range(2)]
    uncs = [np.interp(t, t0, g["uncs"][m]) for m in range(2)]
    tables = {520: (g["moments"], g["t_irf"])}
    sim = {"lengths": list(g["lengths"]), "nx": [nx] * 2, "meas_types": ["TRPL"] * 2, "num_meas": 2}
    prob = _capi.pack_problem(sim, g["inis"], [t] * 2, vals, uncs, model="traps", ini_mode="fluence",
                              irf_convolution=[520, 520], irf_tables=tables)
    params = _capi.pack_params(g["states"][:n], idx, g["units"], model="traps")
    aux = _capi.default_aux(n, 2, [1.0] * 2)
    aux[:, 1, _capi.A_SCALE_SHIFT] = -0.2
    return prob, params, aux, [tables[520]] * 2


def conv_refused_case():
    """traps + IRF at nx = 128 whose second measurement ends at 0.7 of the IRF step: fewer than three
    resampled points, so the convolution is refused (TRPL_ST_CONV_FAIL) for that curve only."""
    g, names, idx, _ = traps128_problem()
    dt = float(np.mean(np.diff(g["t_irf"])))
    t_short = np.linspace(0.0, 0.7 * dt, 6)
    tables = {520: (g["moments"], g["t_irf"])}
    sim = {"lengths": list(g["lengths"]), "nx": [128] * 2, "meas_types": ["TRPL"] * 2, "num_meas": 2}
    prob = _capi.pack_problem(sim, g["inis"], [g["t"], t_short], [g["vals"][0], np.full(6, g["vals"][1][0])],
                              [g["uncs"][0], np.full(6, g["uncs"][1][0])], model="traps", ini_mode="fluence",
                              irf_convolution=[520, 520], irf_tables=tables)
    params = _capi.pack_params(g["states"][:2], idx, g["units"], model="traps")
    return prob, params, _capi.default_aux(2, 2, [1.0] * 2), [tables[520]] * 2


def test_fit_streaming_path_with_scale_shift():
    prob, params, aux = staub_case()
    with_fit = emu_run(prob, params, aux, 0)
    ll, st, ns, cur, fit = with_fit
    assert np.all(np.isfinite(ll))
    n, n_short = check_fit(prob, aux, ll, st, cur, fit)
    assert n == 24 and n_short == 0


def test_fit_force_min_y():
    # a negative shift raises the floor 10**min(vals - shift) into the curves' tails
    prob, params, aux = staub_case(shift=-1.5)
    with_fit = emu_run(prob, params, aux, _capi.OPT_FORCE_MIN_Y)
    ll, st, ns, cur, fit = with_fit
    check_fit(prob, aux, ll, st, cur, fit, force_min_y=True)
    # the floor is in use: some fitted points sit exactly on min(vals) of their curve
    sl = slice(0, int(prob.n_t[0]))
    floor = np.min(prob.vals[sl]) - (-1.5)
    assert np.any(np.abs(fit[:, sl] - (np.log10(10.0 ** floor) - 1.5)) == 0)


def test_fit_traps_irf_nx256():
    prob, params, aux, tables = traps_irf_case()
    with_fit = emu_run(prob, params, aux, 0)
    ll, st, ns, cur, fit = with_fit
    n, n_short = check_fit(prob, aux, ll, st, cur, fit, irf_tables=tables)
    assert n_short == n            # the trim drops the tail of every curve


def test_fit_irf_uneven_times():
    g = np.load(pc.os.path.join(pc.GOLDEN, "traps_irf.npz"))
    t0 = g["t"]
    n = len(t0)
    prob, params, aux, tables = traps_irf_case(nx=128, n=2, times=t0[-1] * (np.arange(n) / (n - 1)) ** 1.4)
    with_fit = emu_run(prob, params, aux, 0)
    ll, st, ns, cur, fit = with_fit
    check_fit(prob, aux, ll, st, cur, fit, irf_tables=tables)


def test_fit_refused_convolution_is_all_nan():
    prob, params, aux, tables = conv_refused_case()
    with_fit = emu_run(prob, params, aux, 0)
    ll, st, ns, cur, fit = with_fit
    assert np.all(st[:, 1] & _capi.ST_CONV_FAIL) and not np.any(st[:, 0] & _capi.ST_CONV_FAIL)
    assert np.all(np.isnan(fit[:, prob.t_off[1]:]))
    check_fit(prob, aux, ll, st, cur, fit, irf_tables=tables)
