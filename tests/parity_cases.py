"""Parity cases shared by the CPU tier (host lock-step build of the kernel source) and the GPU tier
(the CUDA library through its C ABI).  A *backend* is a callable

    backend(prob, params, aux, opts, want_curves) -> (logll[n_sets,n_meas,3], status, nsteps, curves)

What "the truth" is (DESIGN.md section 6).  The reference's LSODA run is not converged once a curve
has decayed a few decades (its default atol = 1e-10 nm^-3 exceeds the densities; tightening it to
1e-14 still leaves errors of atol / excess density, and beyond that SciPy's LSODA stalls - measured,
see DESIGN.md).  Every fixture state is therefore checked against THREE routes that share no time
integrator:
  (A) the integrator under test at rtol = 1e-9 (CPU) / 1e-10 (GPU): self-convergence;
  (B) the reference's algorithm (SciPy LSODA on the bit-exact right-hand side) at rtol 1e-10 /
      atol 1e-14, inside the part of the curve where that run can be accurate (top three decades);
  (C) the linear-regime asymptote: at low injection the reference's equations are linear and every
      curve ends as exp(-lambda t) with lambda an eigenvalue of the reference's Jacobian at
      equilibrium (oracle/excess_model.decay_rates, LAPACK, no time stepping at all).
Tolerances (stated here once, asserted below; RANGE = 14 decades below each curve's first point,
the dynamic range the error control covers - trajectory.h EXCESS_RANGE plus the initial transient):
  CURVE_TOL         = 1e-5   relative per time step, run under test vs route (A), every point of
                             every state within RANGE  (north star: <= 1e-4)
  CURVE_TOL_LSODA   = 1e-5   route (A) vs route (B), top three decades of every curve
  RATE_TOL          = 2e-6   log-slope of a deep single-exponential tail vs route (C)
  CURVE_TOL_DEFAULT = 1e-4   vs the reference at its DEFAULT tolerances, every point within RANGE,
                             up to that run's own distance from route (A) (triangle inequality; no mask)
  LOGLL_TOL         = 1e-6   relative, every state whose converged log-likelihood is > -1e4
                             (north star: <= 1e-6), at three temperatures
"""
import os

import numpy as np

from metrotrpl_b200 import _capi
from oracle import excess_model as exm
from oracle import trpl_oracle as orc

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

CURVE_TOL = 1e-5
CURVE_TOL_LSODA = 1e-5
CURVE_TOL_CLEAN = 1e-6
RATE_TOL = 2e-6
CURVE_TOL_DEFAULT = 1e-4
LOGLL_TOL = 1e-6
RANGE_DECADES = 14.0
LOGLL_FLOOR = -1e4          # states below this are certain rejections: decision parity only


def staub_problem():
    g = np.load(os.path.join(GOLDEN, "staub6.npz"))
    names = [str(n) for n in g["names"]]
    idx = {n: i for i, n in enumerate(names)}
    t = g["t"]
    sim = {"lengths": list(g["lengths"]), "nx": [int(g["nx"])] * 6, "meas_types": ["TRPL"] * 6,
           "num_meas": 6}
    prob = _capi.pack_problem(sim, g["ini"], [t] * 6, list(g["vals"]), list(g["uncs"]))
    params = _capi.pack_params(g["states"], idx, g["units"])
    aux = _capi.default_aux(params.shape[0], 6, [float(g["sigma"])] * 6, temps=tuple(g["temps"]))
    return g, prob, params, aux


def real3_problem():
    """configs[0] on the reference's real data (tools/make_golden.py gen_real3)."""
    g = np.load(os.path.join(GOLDEN, "staub_real3.npz"))
    names = [str(n) for n in g["names"]]
    idx = {n: i for i, n in enumerate(names)}
    n_t = g["n_t"]
    times = [g["t"][m, :n_t[m]] for m in range(3)]
    vals = [g["vals"][m, :n_t[m]] for m in range(3)]
    uncs = [g["uncs"][m, :n_t[m]] for m in range(3)]
    sim = {"lengths": list(g["lengths"]), "nx": [int(g["nx"])] * 3, "meas_types": ["TRPL"] * 3, "num_meas": 3}
    prob = _capi.pack_problem(sim, g["ini"], times, vals, uncs)
    params = _capi.pack_params(g["states"], idx, g["units"])
    aux = _capi.default_aux(params.shape[0], 3, [float(g["sigma"])] * 3, temps=tuple(g["temps"]))
    return g, prob, params, aux, times, vals, uncs


def _model_args(state, units, idx, length, nx):
    s = np.asarray(state, dtype=float) * units
    lam = orc.Q_C / (s[idx["eps"]] * orc.EPS0)
    return (nx, length / nx, s[idx["n0"]], s[idx["p0"]], s[idx["mu_n"]], s[idx["mu_p"]], s[idx["ks"]],
            s[idx["Cn"]], s[idx["Cp"]], s[idx["Sf"]], s[idx["Sb"]], s[idx["tauN"]], s[idx["tauP"]], lam,
            s[idx["Tm"]])


def check_against_converged(backend, g, prob, params, aux, times, vals, uncs, rtol=1e-7, tight_rtol=1e-9,
                            pl_lsoda_tight=None, pl_default=None, min_tails=3, curve_tol=CURVE_TOL, truth_backend=None):
    """Every state of a fixture against the three truth routes of the module docstring."""
    names = [str(n) for n in g["names"]]
    idx = {n: i for i, n in enumerate(names)}
    nS, nM = params.shape[0], len(times)
    sigma = float(g["sigma"])
    ll, status, nsteps, curves = backend(prob, params, aux, _capi.make_opts(RTOL=rtol), True)
    _, _, ns_t, curves_t = (truth_backend or backend)(prob, params, aux, _capi.make_opts(RTOL=tight_rtol), True)
    off = np.concatenate([[0], np.cumsum([len(t) for t in times])])
    cur = [[curves[s, off[m]:off[m + 1]] for m in range(nM)] for s in range(nS)]
    tru = [[curves_t[s, off[m]:off[m + 1]] for m in range(nM)] for s in range(nS)]
    rep = {"rtol": rtol, "truth_rtol": tight_rtol}
    worst = {"curve": 0.0, "lsoda": 0.0, "default_excess": 0.0, "rate": 0.0}
    ref_default_dev = np.zeros(nS)
    n_tails = 0
    for s in range(nS):
        for m in range(nM):
            T, c = tru[s][m], cur[s][m]
            with np.errstate(all="ignore"):
                in_range = T >= 10.0 ** (-RANGE_DECADES) * T[0]
                e = np.where(in_range, np.abs(c / T - 1), 0.0)
            worst["curve"] = max(worst["curve"], float(e.max()))
            assert e.max() <= curve_tol * max(1.0, rtol / 1e-7), (s, m, e.max())
            if pl_lsoda_tight is not None:
                B = pl_lsoda_tight[s][m][:len(T)]
                top = B >= 1e-3 * B[0]
                eb = np.abs(T[top] / B[top] - 1).max()
                worst["lsoda"] = max(worst["lsoda"], float(eb))
                assert eb <= CURVE_TOL_LSODA, (s, m, eb)
            if pl_default is not None:
                D = pl_default[s][m][:len(T)]
                with np.errstate(all="ignore"):
                    ok = in_range & (D > 0)
                    # log ratios, so that the triangle inequality is exact however far the
                    # reference's own run has drifted (it reaches the min_y floor decades early)
                    d_ref = np.where(ok, np.abs(np.log(D) - np.log(T)), 0.0)  # the reference's own solver error
                    d_us = np.where(ok, np.abs(np.log(c) - np.log(D)), 0.0)
                ref_default_dev[s] = max(ref_default_dev[s], float(d_ref.max()))
                excess = float((d_us - d_ref).max())
                worst["default_excess"] = max(worst["default_excess"], excess)
                assert excess <= CURVE_TOL_DEFAULT, (s, m, excess)
            # route (C): a deep, single-exponential tail decays at an eigenvalue of the reference's
            # Jacobian at equilibrium
            t = times[m]
            with np.errstate(all="ignore"):
                k = np.where((T < 1e-8 * T[0]) & (T > 1e-12 * T[0]))[0]
            if len(k) >= 6:
                h = len(k) // 2
                def slope(i, j, y=T):
                    return -(np.log(y[j]) - np.log(y[i])) / (t[j] - t[i])
                s1, s2 = slope(k[0], k[h]), slope(k[h], k[-1])
                if abs(s1 / s2 - 1) <= 2e-7:              # one mode left
                    rates = exm.decay_rates(*_model_args(g["states"][s], g["units"], idx,
                                                         float(g["lengths"][m]), int(g["nx"])))
                    sl_t, sl_c = slope(k[0], k[-1]), slope(k[0], k[-1], c)
                    dev_t = np.abs(sl_t / rates - 1).min()
                    dev_c = np.abs(sl_c / rates - 1).min()
                    worst["rate"] = max(worst["rate"], float(dev_t), float(dev_c))
                    assert dev_t <= RATE_TOL and dev_c <= RATE_TOL, (s, m, sl_t, sl_c, dev_t, dev_c)
                    n_tails += 1
    assert n_tails >= min_tails, n_tails
    rep["max_curve_err_vs_converged_within_range"] = worst["curve"]
    rep["max_converged_vs_lsoda_tight_top3decades"] = worst["lsoda"]
    rep["max_excess_over_reference_default_error"] = worst["default_excess"]
    rep["deep_tails_checked_against_jacobian_eigenvalues"] = n_tails
    rep["max_decay_rate_rel_err"] = worst["rate"]
    # log-likelihood: every state above LOGLL_FLOOR, three temperatures, against the likelihood of
    # the converged curves (the oracle's restatement of one_sim_likelihood, pinned to the reference)
    rows = []
    worst_ll = 0.0
    for s in range(nS):
        conv = [sum(orc.curve_loglik(tru[s][m], times[m], times[m], vals[m], uncs[m], sigma, T=float(temp))
                    for m in range(nM)) for temp in g["temps"]]
        ours = [ll[s, :, k].sum() for k in range(3)]
        if conv[0] > LOGLL_FLOOR:
            rel = max(abs(ours[k] / conv[k] - 1) for k in range(3))
            ref_rel = abs(float(g["logll"][s]) / conv[0] - 1)
            rows.append((s, float(conv[0]), float(ours[0]), float(rel), float(g["logll"][s]), float(ref_rel),
                         float(ref_default_dev[s])))
            worst_ll = max(worst_ll, rel)
            assert rel <= LOGLL_TOL * max(1.0, rtol / 1e-7), (s, conv, ours, rel)
            assert np.all((status[s] & ~_capi.ST_FLOORED) == 0)
        else:
            # certain rejection for everybody: only the decision is compared
            assert ours[0] < 0.999 * LOGLL_FLOOR, (s, conv[0], ours[0])
            assert float(g["logll"][s]) < 0.5 * LOGLL_FLOOR, (s, g["logll"][s])
    rep["logll_rows_[state,converged,ours,rel,reference_default,ref_rel,ref_curve_dev]"] = rows
    rep["max_logll_rel_vs_converged"] = worst_ll
    rep["states_above_floor"] = len(rows)
    rep["mean_steps"] = float(nsteps[..., 0].mean())
    rep["mean_rejected"] = float(nsteps[..., 1].mean())
    rep["mean_steps_truth_run"] = float(ns_t[..., 0].mean())
    return rep


def check_staub(backend, rtol=1e-7, tight_rtol=1e-9, **kw):
    """The six-curve staub example (Inputs/mcmc0.txt grid and initial conditions), 17 states."""
    g, prob, params, aux = staub_problem()
    t = g["t"]
    return check_against_converged(backend, g, prob, params, aux, [t] * 6, list(g["vals"]), list(g["uncs"]),
                                   rtol=rtol, tight_rtol=tight_rtol, pl_lsoda_tight=g["pl_tight"],
                                   pl_default=g["pl_default"], min_tails=8, **kw)


def check_real3(backend, rtol=1e-7, tight_rtol=1e-9, **kw):
    """configs[0] on the reference's real measurement (values and uncertainties of
    Inputs/real_staub_aug_corr_renoised.csv), 17 states."""
    g, prob, params, aux, times, vals, uncs = real3_problem()
    n_t = g["n_t"]
    D = [[g["pl_default"][s, m, :n_t[m]] for m in range(3)] for s in range(params.shape[0])]
    return check_against_converged(backend, g, prob, params, aux, times, vals, uncs, rtol=rtol,
                                   tight_rtol=tight_rtol, pl_default=D, min_tails=3, **kw)


def _known_units():
    names = ["n0", "p0", "mu_n", "mu_p", "ks", "Cn", "Cp", "Tm", "Sf", "Sb", "tauN", "tauP", "eps", "m"]
    uc = {"n0": 1e-21, "p0": 1e-21, "mu_n": 1e5, "mu_p": 1e5, "ks": 1e12, "Sf": 1e-2, "Sb": 1e-2}
    units = np.array([uc.get(n, 1) for n in names], dtype=float)
    return names, units, {n: i for i, n in enumerate(names)}


BASE = {"n0": 0, "p0": 0, "mu_n": 0, "mu_p": 0, "ks": 1e-11, "Sf": 0, "Sb": 0, "Cn": 0, "Cp": 0,
        "Tm": 300, "tauN": 1e99, "tauP": 1e99, "eps": 10, "m": 1}


def _run_known(backend, guess, lengths, nxs, mtypes, ini, times, vals, uncs, sigma, rtol=1e-5,
               atol=1e-8, flags=0, want_curves=False):
    names, units, idx = _known_units()
    sim = {"lengths": lengths, "nx": nxs, "meas_types": mtypes, "num_meas": len(lengths)}
    prob = _capi.pack_problem(sim, ini, times, vals, uncs)
    state = np.array([[guess[n] for n in names]], dtype=float)
    params = _capi.pack_params(state, idx, units)
    aux = _capi.default_aux(1, len(lengths), [sigma[m] for m in mtypes])
    opts = _capi.make_opts(RTOL=rtol, ATOL=atol, flags=flags)
    ll, st, ns, cur = backend(prob, params, aux, opts, want_curves)
    return ll[0, :, 0], st[0], cur


def check_known_answers(backend):
    """The five cases of the reference's Tests/test_eval_trial_move.py, at the tolerances that file
    passes (rtol=1e-5, atol=1e-8) and with its own acceptance criteria."""
    g = np.load(os.path.join(GOLDEN, "known_answers.npz"))
    t100 = np.linspace(0, 100, 1001)
    ini2 = np.array([1e15 * np.ones(128), 1e16 * np.ones(128)])
    flat = [np.ones(1001) * 23] * 2
    tiny = [np.ones(1001) * 1e-99] * 2
    out = {}
    # test_run_iter (Tests/test_eval_trial_move.py:21-80)
    per, st, cur = _run_known(backend, BASE, [2000, 2000], [128, 128], ["TRPL", "TRPL"], ini2,
                              [t100, t100], flat, tiny, {"TRPL": 1.0}, want_curves=True)
    np.testing.assert_almost_equal(per.sum(), np.sum([-59340.105083, -32560.139058]), decimal=0)
    assert abs(per.sum() / float(g["run_iter"]) - 1) < 1e-5
    np.testing.assert_allclose(cur[0, :1001], g["run_iter_pl0_tight"], rtol=2e-5)
    out["run_iter"] = float(per.sum())
    # test_run_iter_cutoff (:145-208)
    t50 = np.linspace(0, 50, 501)
    per, st, _ = _run_known(backend, BASE, [2000, 2000], [128, 128], ["TRPL", "TRPL"], ini2, [t50, t50],
                            [np.ones(501) * 23] * 2, [np.ones(501) * 1e-99] * 2, {"TRPL": 1.0})
    np.testing.assert_almost_equal(per.sum(), -45982, decimal=0)
    assert abs(per.sum() / float(g["run_iter_cutoff"]) - 1) < 1e-5
    # test_run_iter_mixed_types (:281-341): TRPL + TRTS
    mixed = dict(BASE, mu_n=0.01, mu_p=0.01)
    ini3 = np.array([1e15 * np.ones(128), 1e15 * np.ones(128)])
    per, st, cur = _run_known(backend, mixed, [2000, 2000], [128, 128], ["TRPL", "TRTS"], ini3,
                              [t100, t100], [np.ones(1001) * 23, np.ones(1001) * -2], tiny,
                              {"TRPL": 1.0, "TRTS": 10.0}, want_curves=True)
    np.testing.assert_almost_equal(per.sum(), np.sum([-59340.105083, -517.98]), decimal=0)
    assert abs(per.sum() / float(g["mixed_types"]) - 1) < 1e-5
    np.testing.assert_allclose(cur[0, 1001:], g["mixed_trts_tight"], rtol=2e-5)
    out["mixed"] = float(per.sum())
    # test_run_iter_depletion (:82-143): force_min_y makes the two likelihoods comparable
    dep = dict(BASE, n0=1e8, p0=1e17, ks=1e-13, tauN=4, tauP=4)
    vals = [np.log10(2e14 * np.exp(-t100 / 8))]
    ini1 = np.array([1e15 * np.ones(128)])
    lls = []
    names, units, idx = _known_units()
    sim1 = {"lengths": [2000], "nx": [128], "meas_types": ["TRPL"], "num_meas": 1}
    for tau in (4, 4.01):
        d = dict(dep, tauN=tau, tauP=tau)
        per, st, cur = _run_known(backend, d, [2000], [128], ["TRPL"], ini1, [t100], vals,
                                  [np.ones(1001) * 1e-99], {"TRPL": 1.0}, rtol=1e-7,
                                  flags=_capi.OPT_FORCE_MIN_Y)
        lls.append(per.sum())
        # The reference's own number at the test's loose tolerances (rtol=1e-5/atol=1e-8, fixture
        # "depletion_4" = -1620.88) is solver noise below atol; as its tolerances tighten it converges
        # (-1424.50 at 1e-7/1e-10, -1392.3403 at 1e-11/1e-18).  Parity is against that limit,
        # computed here with the pinned oracle (same LSODA, same RHS).
        state = np.array([d[n] for n in names], dtype=float)
        want, _ = orc.state_loglik(state, sim1, ini1, [t100], vals, [np.ones(1001) * 1e-99], idx, units,
                                   {"TRPL": 1.0}, rtol=1e-11, atol=1e-18, force_min_y=True)
        assert abs(per.sum() / want - 1) < 1e-6, (per.sum(), want)
    assert lls[1] > lls[0]                       # Tests/test_eval_trial_move.py:143
    # curve-level parity in the converged part of the depleting curve
    ref = g["depletion_pl_tight"]
    okm = ref > 1e-6 * ref[0]
    d = dict(dep)
    per, st, cur = _run_known(backend, d, [2000], [128], ["TRPL"], ini1, [t100], vals,
                              [np.ones(1001) * 1e-99], {"TRPL": 1.0}, rtol=1e-7, want_curves=True)
    np.testing.assert_allclose(cur[0][okm], ref[okm], rtol=1e-5)
    out["depletion"] = [float(x) for x in lls]
    return out


def check_analytic(backend):
    """Closed-form limits, in the spirit of the reference's Tests/test_forward_solver.py."""
    names, units, idx = _known_units()
    nx, L = 100, 1000.0
    t = np.linspace(0, 10, 101)
    sim = {"lengths": [L], "nx": [nx], "meas_types": ["TRPL"], "num_meas": 1}
    out = {}
    # (a) radiative only, high injection, uniform: dN/dt = -ks N^2
    N0 = 1e17
    prob = _capi.pack_problem(sim, [N0 * np.ones(nx)], [t], None, None)
    guess = dict(BASE, ks=1e-10)
    st = np.array([[guess[n] for n in names]], dtype=float)
    aux = _capi.default_aux(1, 1, [1.0])
    opts = _capi.make_opts(RTOL=1e-8, flags=_capi.OPT_NO_LIKELIHOOD)
    _, s, ns, cur = backend(prob, _capi.pack_params(st, idx, units), aux, opts, True)
    ks = 1e-10 * 1e12
    n0m = N0 * 1e-21
    Nt = n0m / (1 + ks * n0m * t)
    expect = ks * Nt ** 2 * L * 1e23
    np.testing.assert_allclose(cur[0], expect, rtol=2e-7)
    # (b) SRH only, tauN = tauP = 1 ns, high injection: lifetime tauN + tauP (test_solver_HI_srh)
    guess = dict(BASE, ks=1e-20, tauN=1.0, tauP=1.0)
    st = np.array([[guess[n] for n in names]], dtype=float)
    prob = _capi.pack_problem(sim, [1e10 * np.ones(nx)], [t], None, None)
    _, s, ns, cur = backend(prob, _capi.pack_params(st, idx, units), aux, opts, True)
    Nt = 1e10 * 1e-21 * np.exp(-t / 2.0)
    expect = 1e-20 * 1e12 * Nt ** 2 * L * 1e23
    np.testing.assert_allclose(cur[0], expect, rtol=2e-7)
    # (c) diffusion only: carriers are conserved, so the photoconductivity is constant in time
    #     while the PL of a non-uniform profile relaxes to that of the mean (test_solver_diffusion)
    sim2 = {"lengths": [L, L], "nx": [nx, nx], "meas_types": ["TRTS", "TRPL"], "num_meas": 2}
    prof = np.logspace(14, 8, nx)
    t2 = np.linspace(0, 2000, 21)
    prob = _capi.pack_problem(sim2, [prof, prof], [t2, t2], None, None)
    g0 = dict(BASE, mu_n=100, mu_p=100, ks=0.0)       # no recombination at all: TRTS check
    g1 = dict(BASE, mu_n=100, mu_p=100, ks=1e-11)     # weak radiative term so that PL is non-zero
    st = np.array([[g0[n] for n in names], [g1[n] for n in names]], dtype=float)
    aux2 = _capi.default_aux(2, 2, [1.0, 1.0])
    _, s, ns, cur = backend(prob, _capi.pack_params(st, idx, units), aux2, opts, True)
    trts = cur[0, :21]
    np.testing.assert_allclose(trts, trts[0], rtol=1e-9)
    expect0 = orc.Q_C * (2 * 100 * 1e5) * np.sum(prof * 1e-21) * (L / nx) * 1e9
    np.testing.assert_allclose(trts[0], expect0, rtol=1e-12)
    assert np.all(cur[0, 21:] == np.finfo(float).tiny)      # ks = 0: PL == 0 -> floored to DBL_MIN
    pl = cur[1, 21:]
    mean = np.mean(prof * 1e-21)
    # ks N^2 recombination is negligible on this time scale (1/(ks N) >> 2000 ns)
    np.testing.assert_allclose(pl[-1], 1e-11 * 1e12 * mean ** 2 * L * 1e23, rtol=2e-3)
    assert pl[0] > 5 * pl[-1]
    out["steps_diffusion"] = ns[0, :, 0].tolist()
    return out


def check_edges(backend):
    """Ragged / degenerate inputs: unequal curve lengths, nx not a multiple of 32, a single time
    point, fluence-mode initial condition (both directions), scale factors and temperatures."""
    names, units, idx = _known_units()
    guess = dict(BASE, n0=1e8, p0=3e15, mu_n=20, mu_p=20, ks=4.8e-11, Cn=4.4e-29, Cp=4.4e-29,
                 Sf=10, Sb=1e3, tauN=511, tauP=871)
    st = np.array([[guess[n] for n in names]], dtype=float)
    params = _capi.pack_params(st, idx, units)
    t_a = np.array([0.0])
    t_b = np.concatenate([[0.0], np.logspace(-1, 2.5, 37)])
    t_c = np.linspace(0, 50, 11)
    sim = {"lengths": [311.0, 500.0, 2000.0], "nx": [40, 64, 50], "meas_types": ["TRPL"] * 3, "num_meas": 3}
    inis = [np.array([2e12, 6e4, 1.0]), np.array([2e12, 6e4, -1.0]), np.array([2e12, 6e4, 1.0])]
    vals = [np.array([17.0]), np.full(38, 16.5), np.full(11, 16.0)]
    uncs = [np.array([0.05]), np.full(38, 0.05), np.full(11, 0.05)]
    prob = _capi.pack_problem(sim, inis, [t_a, t_b, t_c], vals, uncs, ini_mode="fluence")
    aux = _capi.default_aux(1, 3, [1.0] * 3, temps=(1.0, 4.0, 16.0))
    aux[0, 1, _capi.A_SCALE_SHIFT] = 0.3
    opts = _capi.make_opts(RTOL=1e-8)
    ll, s, ns, cur = backend(prob, params, aux, opts, True)
    # oracle on the same three curves
    for m in range(3):
        g = orc.Grid(sim["lengths"][m], sim["nx"][m], [t_a, t_b, t_c][m], 4)
        ref = orc.simulate(inis[m], g, st[0], idx, units=units, ini_mode="fluence", RTOL=1e-10,
                           ATOL=1e-16)
        mine = cur[0, prob.t_off[m]:prob.t_off[m] + prob.n_t[m]]
        np.testing.assert_allclose(mine, ref, rtol=2e-6)
        for k, temp in enumerate((1.0, 4.0, 16.0)):
            shift = 0.3 if m == 1 else 0.0
            want = orc.curve_loglik(ref, g.tSteps, g.tSteps, vals[m], uncs[m], 1.0, T=temp,
                                    scale_shift=shift)
            assert abs(ll[0, m, k] - want) <= 2e-6 * abs(want) + 1e-12
    # reversing the illumination side of a symmetric-contact film gives the same PL
    sim_s = {"lengths": [400.0, 400.0], "nx": [33, 33], "meas_types": ["TRPL"] * 2, "num_meas": 2}
    gsym = dict(guess, Sb=10)
    st2 = np.array([[gsym[n] for n in names]], dtype=float)
    prob = _capi.pack_problem(sim_s, [inis[0], inis[1]], [t_c, t_c], None, None, ini_mode="fluence")
    _, s, ns, cur = backend(prob, _capi.pack_params(st2, idx, units), _capi.default_aux(1, 2, [1.0] * 2),
                            _capi.make_opts(RTOL=1e-8, flags=_capi.OPT_NO_LIKELIHOOD), True)
    np.testing.assert_allclose(cur[0, :11], cur[0, 11:], rtol=1e-7)
    # every nodes-per-lane instantiation, with padding: nx = 16 (1/lane), 200 (two-warp team, 4/lane), 'traps' at 100 (4/lane)
    for nx, model in ((16, "std"), (200, "std"), (100, "traps")):
        names_m = names + (["kC", "Nt", "tauE"] if model == "traps" else [])
        units_m = np.concatenate([units, [1e12, 1e-21, 1.0]]) if model == "traps" else units
        idx_m = {n: i for i, n in enumerate(names_m)}
        gm = dict(guess, kC=1e-8, Nt=1e15, tauE=50.0)
        stm = np.array([[gm[n] for n in names_m]], dtype=float)
        simn = {"lengths": [500.0], "nx": [nx], "meas_types": ["TRPL"], "num_meas": 1}
        prob = _capi.pack_problem(simn, [inis[0]], [t_c], None, None, model=model, ini_mode="fluence")
        _, s, ns, cur = backend(prob, _capi.pack_params(stm, idx_m, units_m, model=model),
                                _capi.default_aux(1, 1, [1.0]),
                                _capi.make_opts(RTOL=1e-8, flags=_capi.OPT_NO_LIKELIHOOD), True)
        g = orc.Grid(500.0, nx, t_c, 4)
        ref = orc.simulate(inis[0], g, stm[0], idx_m, units=units_m, model=model, ini_mode="fluence",
                           RTOL=1e-10, ATOL=1e-16)
        np.testing.assert_allclose(cur[0], ref, rtol=2e-6)
    return True


def check_traps_irf(backend, curve_tol=CURVE_TOL_CLEAN):
    """BASELINE configs[3]: trap-assisted model + IRF convolution (IRFs/irf_520nm.csv), nx=256,
    fluence-mode initial condition, stiff capture.  Curves against the reference at tight
    tolerances; likelihood (resample -> convolve -> max-shift -> trim -> log residuals) against the
    oracle's restatement of laplace.py run on the converged reference curves and on our own curves."""
    g = np.load(os.path.join(GOLDEN, "traps_irf.npz"))
    names = [str(n) for n in g["names"]]
    idx = {n: i for i, n in enumerate(names)}
    t = g["t"]
    nx = int(g["nx"])
    tables = {520: (g["moments"], g["t_irf"])}
    sim = {"lengths": list(g["lengths"]), "nx": [nx] * 2, "meas_types": ["TRPL"] * 2, "num_meas": 2}
    prob = _capi.pack_problem(sim, g["inis"], [t] * 2, list(g["vals"]), list(g["uncs"]), model="traps",
                              ini_mode="fluence", irf_convolution=[520, 520], irf_tables=tables)
    params = _capi.pack_params(g["states"], idx, g["units"], model="traps")
    nS = params.shape[0]
    aux = _capi.default_aux(nS, 2, [1.0] * 2)
    ll, st, ns, cur = backend(prob, params, aux, _capi.make_opts(RTOL=1e-7), True)
    cur = cur.reshape(nS, 2, len(t))
    rep = {}
    e_t = np.abs(cur / g["pl_tight"] - 1).max()
    rep["curve_err_vs_tight"] = float(e_t)
    assert e_t <= curve_tol, e_t
    # the reference at its default tolerances is itself off by up to 1.5e-3 on the stiff states
    ref_ok = np.abs(g["pl_default"] / g["pl_tight"] - 1) <= 5e-5
    e_d = np.where(ref_ok, np.abs(cur / g["pl_default"] - 1), 0).max()
    rep["curve_err_vs_default_where_ref_converged"] = float(e_d)
    rep["frac_ref_converged"] = float(ref_ok.mean())
    assert e_d <= CURVE_TOL_DEFAULT
    worst_conv, worst_chain, worst_def = 0.0, 0.0, 0.0
    for s in range(nS):
        ours = ll[s, :, 0].sum()
        conv = sum(orc.curve_loglik(g["pl_tight"][s, m], t, t, g["vals"][m], g["uncs"][m], 1.0,
                                    irf_table=tables[520]) for m in range(2))
        chain = sum(orc.curve_loglik(cur[s, m], t, t, g["vals"][m], g["uncs"][m], 1.0,
                                     irf_table=tables[520]) for m in range(2))
        worst_conv = max(worst_conv, abs(ours / conv - 1))
        worst_chain = max(worst_chain, abs(ours / chain - 1))
        worst_def = max(worst_def, abs(ours / g["logll"][s] - 1))
    rep["logll_rel_vs_converged_ref"] = worst_conv
    rep["logll_rel_irf_chain_only"] = worst_chain
    rep["logll_rel_vs_default_ref"] = worst_def
    assert worst_chain <= 1e-12      # the convolution/trim/likelihood chain itself is exact to rounding
    assert worst_conv <= LOGLL_TOL
    assert worst_def <= 5e-5         # the reference's own solver error on these states is 1.2e-5
    assert np.all(st == 0)
    rep["steps"] = ns[..., 0].tolist()
    return rep


def check_irf_uneven_times(backend):
    """The IRF pass on measurement times that are NOT equally spaced (denser early, and a jittered
    grid): resampling and trimming locate their interval by a guess from the mean spacing and fall
    back to a search where the guess misses.  Our likelihood against the oracle's restatement of
    laplace.py applied to our own curves: exact to rounding, as on the even grid."""
    g = np.load(os.path.join(GOLDEN, "traps_irf.npz"))
    names = [str(n) for n in g["names"]]
    idx = {n: i for i, n in enumerate(names)}
    t0 = g["t"]
    nx = int(g["nx"])
    tables = {520: (g["moments"], g["t_irf"])}
    sim = {"lengths": list(g["lengths"]), "nx": [nx] * 2, "meas_types": ["TRPL"] * 2, "num_meas": 2}
    rng = np.random.default_rng(3)
    n = len(t0)
    grids = {"power": t0[-1] * (np.arange(n) / (n - 1)) ** 1.4,
             "jitter": np.concatenate([[0.0], np.sort(t0[1:-1] + rng.uniform(-0.1, 0.1, n - 2)), [t0[-1]]])}
    rep = {}
    params = _capi.pack_params(g["states"][:2], idx, g["units"], model="traps")
    aux = _capi.default_aux(2, 2, [1.0] * 2)
    for name, t in grids.items():
        vals = [np.interp(t, t0, g["vals"][m]) for m in range(2)]
        uncs = [np.interp(t, t0, g["uncs"][m]) for m in range(2)]
        prob = _capi.pack_problem(sim, g["inis"], [t] * 2, vals, uncs, model="traps", ini_mode="fluence",
                                  irf_convolution=[520, 520], irf_tables=tables)
        ll, st, ns, cur = backend(prob, params, aux, _capi.make_opts(RTOL=1e-7), True)
        cur = cur.reshape(2, 2, n)
        worst = 0.0
        for s_ in range(2):
            chain = sum(orc.curve_loglik(cur[s_, m], t, t, vals[m], uncs[m], 1.0, irf_table=tables[520])
                        for m in range(2))
            worst = max(worst, abs(ll[s_, :, 0].sum() / chain - 1))
        assert np.all(st == 0) and worst <= 1e-12, (name, worst, st)
        rep[name] = worst
    return rep


def check_explicit_path(backend):
    """Non-stiff trajectories (no transport: the mobility-free cases of the reference's unit tests)
    are classified at t = 0 and integrated by the embedded explicit Runge-Kutta pair; the result must
    agree with the Rosenbrock path and with the converged reference, in fewer and cheaper steps."""
    names, units, idx = _known_units()
    t = np.linspace(0, 100, 1001)
    sim = {"lengths": [2000, 2000], "nx": [128, 128], "meas_types": ["TRPL", "TRTS"], "num_meas": 2}
    ini = np.array([1e15 * np.ones(128), 3e15 * np.exp(-np.arange(128) / 40.0)])
    guess = dict(BASE, n0=1e8, p0=1e17, ks=1e-13, tauN=4, tauP=6, Cn=1e-29, Cp=1e-29)
    stiff = dict(guess, mu_n=20, mu_p=20, Sf=10, Sb=10)
    st = np.array([[guess[n] for n in names], [stiff[n] for n in names]], dtype=float)
    params = _capi.pack_params(st, idx, units)
    prob = _capi.pack_problem(sim, ini, [t, t], None, None)
    aux = _capi.default_aux(2, 2, [1.0, 1.0])
    base = _capi.OPT_NO_LIKELIHOOD
    _, s_auto, n_auto, c_auto = backend(prob, params, aux, _capi.make_opts(RTOL=1e-8, flags=base), True)
    _, s_ros, n_ros, c_ros = backend(prob, params, aux, _capi.make_opts(RTOL=1e-8, flags=base | _capi.OPT_NO_EXPLICIT), True)
    assert np.all(s_auto[0] & _capi.ST_EXPLICIT) and not np.any(s_auto[1] & _capi.ST_EXPLICIT)
    assert not np.any(s_ros & _capi.ST_EXPLICIT)
    # same stiff trajectories either way, bit for bit
    np.testing.assert_array_equal(c_auto[1], c_ros[1])
    ok = c_ros[0] > 1e-6 * c_ros[0].max()
    np.testing.assert_allclose(c_auto[0][ok], c_ros[0][ok], rtol=2e-7)
    assert n_auto[0, :, 0].sum() < 0.7 * n_ros[0, :, 0].sum()
    for m, meas in enumerate(("TRPL", "TRTS")):
        g = orc.Grid(2000, 128, t, 4)
        ref = orc.simulate(ini[m], g, st[0], idx, meas=meas, units=units, RTOL=1e-11, ATOL=1e-18)
        mine = c_auto[0, m * 1001:(m + 1) * 1001]
        okm = ref > 1e-6 * ref[0]
        np.testing.assert_allclose(mine[okm], ref[okm], rtol=2e-6)
    return {"explicit_steps": n_auto[0, :, 0].tolist(), "rosenbrock_steps": n_ros[0, :, 0].tolist()}


def check_team_grids(backend):
    """Grids of 129..256 nodes run on a team of two warps per trajectory (csrc/team_kernels.cu: 64
    lanes x 4 nodes, 6-level reduction, values crossing the warp boundary through a mailbox), grids of
    257..512 nodes on a team of four (team4_kernels.cu: 128 lanes, 7 levels, three boundaries).  Both
    models, padding-free (nx = 256, 512) and padded (nx = 160, 200, 400) grids, TRPL and TRTS, the stiff
    Rosenbrock path and the explicit Runge-Kutta path, against the oracle's LSODA at tight tolerances."""
    names, units, idx = _known_units()
    t = np.linspace(0, 60, 121)
    out = {}
    base = dict(BASE, n0=1e8, p0=3e15, ks=4.8e-11, tauN=511, tauP=871, Cn=4.4e-29, Cp=4.4e-29)
    stiff = dict(base, mu_n=20, mu_p=20, Sf=10, Sb=10)
    nonstiff = dict(base, mu_n=0, mu_p=0, Sf=0, Sb=0, tauN=4, tauP=6, p0=1e17)
    for nx, model in ((256, "std"), (160, "std"), (200, "traps"), (256, "traps"), (400, "std"), (512, "traps")):
        names_m = names + (["kC", "Nt", "tauE"] if model == "traps" else [])
        units_m = np.concatenate([units, [1e12, 1e-21, 1.0]]) if model == "traps" else units
        idx_m = {n: i for i, n in enumerate(names_m)}
        x = (np.arange(nx) + 0.5) * (1000.0 / nx)
        ini = np.array([2e16 * np.exp(-x / 150.0), 5e15 * np.ones(nx)])
        rows = [dict(stiff, kC=1e-8, Nt=1e15, tauE=50.0)]
        if model == "std":
            rows.append(dict(nonstiff, kC=1e-8, Nt=1e15, tauE=50.0))
        st = np.array([[r[n] for n in names_m] for r in rows], dtype=float)
        sim = {"lengths": [1000.0, 1000.0], "nx": [nx, nx], "meas_types": ["TRPL", "TRTS"], "num_meas": 2}
        prob = _capi.pack_problem(sim, ini, [t, t], None, None, model=model)
        _, s, ns, cur = backend(prob, _capi.pack_params(st, idx_m, units_m, model=model),
                                _capi.default_aux(len(rows), 2, [1.0, 1.0]),
                                _capi.make_opts(RTOL=1e-8, flags=_capi.OPT_NO_LIKELIHOOD), True)
        assert not np.any(s & 7), s
        if model == "std":
            assert not np.any(s[0] & _capi.ST_EXPLICIT) and np.all(s[1] & _capi.ST_EXPLICIT), s
        worst = 0.0
        for r in range(len(rows)):
            for m, meas in enumerate(("TRPL", "TRTS")):
                g = orc.Grid(1000.0, nx, t, 4)
                ref = orc.simulate(ini[m], g, st[r], idx_m, meas=meas, units=units_m, model=model,
                                   RTOL=1e-10, ATOL=1e-16)
                mine = cur[r, m * len(t):(m + 1) * len(t)]
                ok = np.abs(ref) > 1e-6 * np.abs(ref[0])
                err = float(np.max(np.abs(mine[ok] / ref[ok] - 1)))
                worst = max(worst, err)
        assert worst < 2e-6, (nx, model, worst)           # measured: 2e-7 (both models, every grid)
        out[f"{model}_nx{nx}"] = {"max_rel_err": worst, "steps": ns[..., 0].tolist()}
    return out


def check_hmax_option(backend):
    """`hmax` (the reference's LSODA max_step, sim_utils.py:17) is accepted and, when asked for,
    imposed as a cap on the step size: same curves, at least t_end / hmax steps."""
    g, prob, params, aux = staub_problem()
    t = g["t"]
    free = _capi.make_opts(RTOL=1e-7)
    capped = _capi.make_opts(RTOL=1e-7, hmax=4.0, honor_hmax=True)
    assert free.hmax == 0.0 and capped.hmax == 4.0
    _, s0, n0, c0 = backend(prob, params[:1], aux[:1], free, True)
    _, s1, n1, c1 = backend(prob, params[:1], aux[:1], capped, True)
    assert np.all(n1[..., 0] >= int(t[-1] / 4.0))
    assert np.all(n0[..., 0] < n1[..., 0])
    np.testing.assert_allclose(c1, c0, rtol=5e-7)
    T = g["pl_tight"][0].reshape(-1)
    np.testing.assert_allclose(c1[0], T, rtol=5e-7)
    return {"free_steps": n0[0, :, 0].tolist(), "capped_steps": n1[0, :, 0].tolist()}


def check_reference_unit_cases(backend):
    """Parameter sets of the reference's remaining unit tests, replayed through the backend:
      Tests/test_forward_solver.py:40-327  test_solver_nothing / LI_SRH / LI_rad / LI_auger
      Tests/test_metropolis.py:199-380     test_solve_depletion / test_solve_traps / test_solve_iniPar
      Tests/test_eval_trial_move.py:210-279 test_run_iter_scale
    The reference's own assertions on N, P are `assert_almost_equal` at 7 decimals on densities of
    1e-11 nm^-3, which any output passes; here each case is held to the closed form its docstring
    names, through the signal the path returns (a radiative probe ks = 1e-20 cm^3/s where the
    reference's parameter set has no readout at all)."""
    names = ["n0", "p0", "mu_n", "mu_p", "ks", "Cn", "Cp", "Sf", "Sb", "tauN", "tauP", "eps", "Tm", "m"]
    uc = {"n0": 1e-21, "p0": 1e-21, "mu_n": 1e5, "mu_p": 1e5, "ks": 1e12, "Cn": 1e33, "Cp": 1e33,
          "Sf": 1e-2, "Sb": 1e-2}
    units = np.array([uc.get(n, 1) for n in names], dtype=float)
    idx = {n: i for i, n in enumerate(names)}
    nx, L = 100, 1000.0
    t = np.linspace(0, 10, 101)
    sim = {"lengths": [L], "nx": [nx], "meas_types": ["TRPL"], "num_meas": 1}
    opts = _capi.make_opts(RTOL=1e-9, flags=_capi.OPT_NO_LIKELIHOOD)
    aux1 = _capi.default_aux(1, 1, [1.0])
    N0 = 1e10 * 1e-21
    base = {"n0": 0, "p0": 0, "mu_n": 0, "mu_p": 0, "ks": 0, "Sf": 0, "Sb": 0, "Cn": 0, "Cp": 0,
            "tauN": 1e99, "tauP": 1e99, "eps": 10, "Tm": 300, "m": 0}
    out = {}

    def pl_of(guess, ini=None, tt=t, model="std", extra_names=(), extra_units=(), min_y=None, meas="TRPL",
              ini_mode="density", length=L):
        nm = names + list(extra_names)
        un = np.concatenate([units, np.array(extra_units, dtype=float)]) if extra_names else units
        ix = {n: i for i, n in enumerate(nm)}
        st = np.array([[guess[n] for n in nm]], dtype=float)
        sm = {"lengths": [length], "nx": [nx], "meas_types": [meas], "num_meas": 1}
        prob = _capi.pack_problem(sm, [1e10 * np.ones(nx) if ini is None else ini], [tt], None, None, model=model,
                                  ini_mode=ini_mode, min_y=min_y)
        _, s, ns, cur = backend(prob, _capi.pack_params(st, ix, un, model=model), aux1, opts, True)
        return cur[0], s[0], ns[0]

    probe = 1e-20 * 1e12                  # ks of the radiative probe in model units
    # test_solver_nothing (:40-84): no process at all; ks = 0 means no PL: the curve is min_y throughout
    cur, s, _ = pl_of(base)
    assert np.all(cur == np.finfo(float).tiny)
    cur, s, _ = pl_of(dict(base, ks=1e-20))
    np.testing.assert_allclose(cur, probe * N0 ** 2 * L * 1e23 * np.ones_like(t), rtol=1e-9)
    # test_solver_LI_SRH (:140-185): tauN = 1, tauP = 1e99, n0 = p0 = 0.  With N = P the SRH rate is
    # N P / (tauN P + tauP N) = N / (1 + 1e99): nothing decays
    cur, s, _ = pl_of(dict(base, ks=1e-20, tauN=1.0))
    np.testing.assert_allclose(cur, probe * N0 ** 2 * L * 1e23 * np.ones_like(t), rtol=1e-9)
    # test_solver_LI_rad (:235-285): p0 = 1 cm^-3, ks = 1e-11, tauN = tauP = 1:
    # dN/dt = -N/2 - ks N^2 (p0 is 1e-10 of N0)  ->  N = N0 e^{-t/2} / (1 + 2 ks N0 (1 - e^{-t/2}))
    ks = 1e-11 * 1e12
    cur, s, _ = pl_of(dict(base, p0=1.0, ks=1e-11, tauN=1.0, tauP=1.0))
    Nt = N0 * np.exp(-t / 2) / (1 + 2 * ks * N0 * (1 - np.exp(-t / 2)))
    np.testing.assert_allclose(cur, ks * Nt ** 2 * L * 1e23, rtol=1e-7)
    # test_solver_LI_auger (:287-327): p0 = 10 cm^-3, Cp = 1e-29: the Auger term is 1e-29 of the SRH one
    cur, s, _ = pl_of(dict(base, p0=10.0, Cp=1e-29, ks=1e-20, tauN=1.0, tauP=1.0))
    np.testing.assert_allclose(cur, probe * (N0 * np.exp(-t / 2)) ** 2 * L * 1e23, rtol=1e-7)
    # test_solve_traps (Tests/test_metropolis.py:270-327): null trap parameters == 'std'; known final density
    t100 = np.linspace(0, 100, 1001)
    tg = dict(base, ks=1e-11, eps=1, kC=0, Nt=0, tauE=1e99)
    ini20 = 1e20 * np.ones(nx)
    cur_t, s, _ = pl_of(tg, ini=ini20, tt=t100, model="traps", extra_names=("kC", "Nt", "tauE"),
                        extra_units=(1e12, 1e-21, 1.0))
    cur_s, s, _ = pl_of(tg | {"m": 0}, ini=ini20, tt=t100)
    out_dN = 0.0009900990095719482                                  # the reference test's constant
    expected = ks * out_dN ** 2 * L * 1e23
    assert abs(cur_t[-1] / expected - 1) < 1e-7                     # reference: 7 decimals of the ratio
    np.testing.assert_allclose(cur_t, cur_s, rtol=1e-9)
    out["traps_final_rel"] = float(cur_t[-1] / expected - 1)
    # test_solve_depletion (:199-268): Grid.min_y truncates the curve (PL and TRTS)
    dg = dict(base, mu_n=1, mu_p=1, ks=2e-10, eps=1)
    ini18 = 1e18 * np.ones(nx)
    full, s, _ = pl_of(dg, ini=ini18, tt=t100)
    assert len(full) == len(t100) and np.all(full > 0)
    PL0 = 2e-10 * 1e12 * (1e18 * 1e-21) ** 2 * L * 1e23
    np.testing.assert_allclose(full[0], PL0, rtol=1e-12)
    cut, s, _ = pl_of(dg, ini=ini18, tt=t100, min_y=[PL0 * 1e-2])
    assert cut.min() >= PL0 * 1e-2 and np.all(cut[-10:] == PL0 * 1e-2)
    first = int(np.argmax(full < PL0 * 1e-2))
    np.testing.assert_allclose(cut[:first], full[:first], rtol=1e-9)
    assert np.all(cut[first:] == PL0 * 1e-2) and (s & _capi.ST_FLOORED)
    TR0 = orc.Q_C * (2 * 1e5) * (1e18 * 1e-21) * L * 1e9
    tr_full, s, _ = pl_of(dg, ini=ini18, tt=t100, meas="TRTS", min_y=[TR0 * 1e-10])
    assert len(tr_full) == len(t100) and tr_full.min() > TR0 * 1e-10
    np.testing.assert_allclose(tr_full[0], TR0, rtol=1e-12)
    tr_cut, s, _ = pl_of(dg, ini=ini18, tt=t100, meas="TRTS", min_y=[TR0 * 1e-1])
    assert tr_cut.min() >= TR0 * 1e-1 and np.all(tr_cut[-10:] == TR0 * 1e-1)
    # test_solve_iniPar (:329-380): [fluence, alpha] (two values, no direction) == the explicit profile
    xs = np.linspace(L / nx / 2, L - L / nx / 2, nx)
    prof = 1e15 * 6e4 * np.exp(-6e4 * xs * 1e-7)
    ig = dict(base, ks=1e-11, eps=1)
    by_vals, s, _ = pl_of(ig, ini=prof, tt=t100)
    by_par, s, _ = pl_of(ig, ini=np.array([1e15, 6e4]), tt=t100, ini_mode="fluence")
    np.testing.assert_allclose(by_par, by_vals, rtol=1e-9)
    # test_run_iter_scale (Tests/test_eval_trial_move.py:210-279): scale factors with constraint
    # groups, through the product's PathCache.pack (group lookup) where the backend is the library
    out["scale"] = check_scale_groups(backend)
    return out


def check_scale_groups(backend):
    """test_run_iter_scale: `_s0`, `_s1` chosen per constraint group ((0,2,4), (1,3,5)) so that both
    curves match the flat measurement: the likelihood is ~0 (reference: 0 to 0 decimals)."""
    from metrotrpl_b200.utils import search_c_grps
    names = ["n0", "p0", "mu_n", "mu_p", "ks", "Cn", "Cp", "Tm", "Sf", "Sb", "tauN", "tauP", "eps", "_s0", "_s1"]
    uc = {"n0": 1e-21, "p0": 1e-21, "mu_n": 1e5, "mu_p": 1e5, "ks": 1e12, "Sf": 1e-2, "Sb": 1e-2}
    units = np.array([uc.get(n, 1) for n in names], dtype=float)
    idx = {n: i for i, n in enumerate(names)}
    guess = {"n0": 0, "p0": 0, "mu_n": 0, "mu_p": 0, "ks": 1e-20, "Sf": 0, "Sb": 0, "Cn": 0, "Cp": 0, "Tm": 300,
             "tauN": 1e99, "tauP": 1e99, "eps": 10, "_s0": 2e-17 ** -1, "_s1": 2e-15 ** -1}
    state = np.array([[guess[n] for n in names]], dtype=float)
    t = np.linspace(0, 100, 1001)
    sim = {"lengths": [2000, 2000], "nx": [128, 128], "meas_types": ["TRPL", "TRPL"], "num_meas": 2}
    ini = np.array([1e15 * np.ones(128), 1e16 * np.ones(128)])
    vals = [np.ones(1001) * 23] * 2
    uncs = [np.ones(1001) * 1e-99] * 2
    spec = (0.02, [0, 1, 2, 3, 4, 5], [(0, 2, 4), (1, 3, 5)])
    prob = _capi.pack_problem(sim, ini, [t, t], vals, uncs)
    params = _capi.pack_params(state, idx, units)
    aux = _capi.default_aux(1, 2, [1.0, 1.0])
    for m in range(2):
        aux[0, m, _capi.A_SCALE_SHIFT] = np.log10(state[0, idx[f"_s{search_c_grps(spec[2], m)}"]])
    ll, st, ns, cur = backend(prob, params, aux, _capi.make_opts(RTOL=1e-5, ATOL=1e-8), True)
    total = ll[0, :, 0].sum()
    np.testing.assert_almost_equal(total, 0, decimal=0)             # the reference's criterion
    sf = {"units": units, "model": "std", "hmax": 4, "rtol": 1e-10, "atol": 1e-18}
    want, _ = orc.state_loglik(state[0], sim, ini, [t, t], vals, uncs, idx, units, {"TRPL": 1.0},
                               rtol=1e-10, atol=1e-18,
                               scale_shifts=[aux[0, m, _capi.A_SCALE_SHIFT] for m in range(2)])
    ll9, _, _, _ = backend(prob, params, aux, _capi.make_opts(RTOL=1e-9), False)
    assert abs(ll9[0, :, 0].sum() - want) <= 1e-6 * abs(want) + 1e-9, (ll9[0, :, 0].sum(), want)
    return {"logll_rtol_1e-5": float(total), "logll_rtol_1e-9": float(ll9[0, :, 0].sum()), "oracle": float(want)}
