"""GPU tier: per-point quantiles of the fitted curves over the sets of a run (trpl_fit_quantiles,
Context.fit_quantiles) bit for bit against np.nanquantile of the downloaded fit, on three kernel
families; the call leaves every output of the run as it was; its refusals; and posterior_predictive
after a metro() run."""
import os
import tempfile
import warnings

import numpy as np
import pytest

from metrotrpl_b200 import _capi
from metrotrpl_b200.metropolis import metro
from metrotrpl_b200.predictive import posterior_predictive
from tests import parity_cases as pc
from tests.test_extrapolation_traps import traps128_problem
from tests.test_fit_curves import traps_irf_case

pytestmark = pytest.mark.gpu

LEVELS = np.array([0.0, 1e-3, 0.025, 0.5, 0.975, 1.0])


@pytest.fixture(scope="module")
def ctx():
    c = _capi.Context(0)
    yield c
    c.close()


def jitter(params, n, names, sigma, seed):
    """n sets: the rows of params in turn, with log10-normal jitter of width sigma on the named slots."""
    rng = np.random.default_rng(seed)
    out = params[np.arange(n) % len(params)].copy()
    for name in names:
        out[:, _capi.PARAM_SLOTS.index(name)] *= 10 ** rng.normal(0, sigma, n)
    return out


def check_run(ctx, prob, params, aux, flags):
    """Run with TRPL_OPT_FIT, then fit_quantiles: equal to NumPy on the downloaded fit, no output of the
    run changed by the call, the same result twice.  Returns (fit, count)."""
    ctx.set_problem(prob)
    ll, st, ns, _ = ctx.loglik_batch(params, aux, _capi.make_opts(RTOL=1e-7, flags=flags | _capi.OPT_FIT))
    fit = ctx.download_fit()
    rng = np.random.default_rng(7)
    for q in (LEVELS, np.sort(rng.random(_capi.MAX_QUANTILES)), [0.5]):
        quant, count = ctx.fit_quantiles(q)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore", RuntimeWarning)
            want = np.nanquantile(fit, q, axis=0, method="linear")
        np.testing.assert_array_equal(quant, want)
        np.testing.assert_array_equal(count, (~np.isnan(fit)).sum(axis=0))
        again = ctx.fit_quantiles(q)
        np.testing.assert_array_equal(again[0], quant)
        np.testing.assert_array_equal(again[1], count)
    ll2, st2, ns2, _ = ctx.download()
    np.testing.assert_array_equal(ll2, ll)
    np.testing.assert_array_equal(st2, st)
    np.testing.assert_array_equal(ns2, ns)
    np.testing.assert_array_equal(ctx.download_fit(), fit)
    # and a run of its own without the call: the same outputs
    ll3, st3, ns3, _ = ctx.loglik_batch(params, aux, _capi.make_opts(RTOL=1e-7, flags=flags | _capi.OPT_FIT))
    np.testing.assert_array_equal(ll3, ll)
    np.testing.assert_array_equal(st3, st)
    np.testing.assert_array_equal(ns3, ns)
    np.testing.assert_array_equal(ctx.download_fit(), fit)
    return fit, count


def test_staub6_rodas4_one_warp_4096_states(ctx):
    g, prob, params, aux = pc.staub_problem()
    p = jitter(params, 4096, ("tauN", "tauP", "Sf", "Sb", "ks"), 0.1, 1)
    aux = np.repeat(aux[:1], 4096, axis=0)
    aux[..., _capi.A_SCALE_SHIFT] = 0.2
    fit, count = check_run(ctx, prob, p, aux, 0)
    assert count.max() == 4096


def test_traps_irf_nx256_two_warp_team_varying_prefix(ctx):
    prob, params, aux, _ = traps_irf_case(nx=256, n=4)
    n = 256
    p = jitter(params, n, ("tauN", "tauP", "Nt", "kC", "tauE", "ks", "Sf", "Sb", "mu_n", "mu_p", "p0"), 1.0, 2)
    fit, count = check_run(ctx, prob, p, np.repeat(aux[:1], n, axis=0), 0)
    n_c = [(~np.isnan(fit[:, prob.t_off[m]:prob.t_off[m] + prob.n_t[m]])).sum(axis=1) for m in range(2)]
    assert any(len(set(c.tolist())) > 1 for c in n_c), "the compared prefix should vary between the states"
    assert np.any((count > 0) & (count < n))


def test_traps_nx128_extrapolation_cta_kernel(ctx):
    g, names, idx, prob = traps128_problem()
    params = _capi.pack_params(g["states"], idx, g["units"], model="traps")
    p = jitter(params, 96, ("tauN", "tauP", "Nt", "kC"), 0.3, 3)
    aux = _capi.default_aux(96, 2, [1.0] * 2)
    check_run(ctx, prob, p, aux, _capi.OPT_EXTRAPOLATION | _capi.OPT_CTA_PER_TRAJ)


def test_refusals(ctx):
    g, prob, params, aux = pc.staub_problem()
    ctx.set_problem(prob)
    ctx.loglik_batch(params[:2], aux[:2], _capi.make_opts())
    with pytest.raises(_capi.TrplError, match=r"the last run did not produce fitted curves \(run with TRPL_OPT_FIT\)"):
        ctx.fit_quantiles([0.5])
    ctx.solve_batch(params[:2], aux[:2], _capi.make_opts())                  # TRPL_OPT_NO_LIKELIHOOD
    with pytest.raises(_capi.TrplError, match=r"did not produce fitted curves \(run with TRPL_OPT_FIT\)"):
        ctx.fit_quantiles([0.5])
    n0 = ctx.launch_count()
    ctx.loglik_batch(params[:2], aux[:2], _capi.make_opts(flags=_capi.OPT_FIT))
    for bad in ([0.5, 1.01], [-0.2], [np.nan]):
        with pytest.raises(_capi.TrplError, match=r"quantile levels must lie in \[0, 1\]"):
            ctx.fit_quantiles(bad)
    for bad in ([], np.linspace(0, 1, _capi.MAX_QUANTILES + 1)):
        with pytest.raises(_capi.TrplError, match="n_q must be in 1..TRPL_MAX_QUANTILES"):
            ctx.fit_quantiles(bad)
    n1 = ctx.launch_count()
    ctx.fit_quantiles([0.5])
    assert ctx.launch_count() == n1 + 1 and n1 > n0                       # refused calls launch nothing


def test_posterior_predictive_after_metro_on_staub6():
    tmp = tempfile.mkdtemp()
    g = np.load(os.path.join(pc.GOLDEN, "staub6.npz"))
    names = [str(n) for n in g["names"]]
    sim = {"lengths": list(g["lengths"]), "nx": [int(g["nx"])] * 6, "meas_types": ["TRPL"] * 6, "num_meas": 6}
    e_data = ([g["t"]] * 6, list(g["vals"]), list(g["uncs"]))
    param_info = {"names": list(names), "active": {n: int(n in ("tauN", "Sf")) for n in names},
                  "unit_conversions": {n: float(u) for n, u in zip(names, g["units"])},
                  "do_log": {n: 1 for n in names}, "prior_dist": {n: (0, np.inf) for n in names},
                  "init_guess": {n: float(v) for n, v in zip(names, g["states"][0])},
                  "trial_move": {n: 0.02 for n in names}}
    MCMC = {"init_cond_path": "x", "measurement_path": "y", "output_path": tmp, "num_iters": 30,
            "solver": ("solveivp",), "model": "std", "ini_mode": "density", "log_y": 1, "checkpoint_freq": 30,
            "rtol": 1e-7, "atol": None, "model_uncertainty": {"TRPL": float(g["sigma"])},
            "parallel_tempering": [1.0, 1.0, 2.0, 4.0], "temper_freq": 5}
    ms = metro(sim, g["ini"], e_data, MCMC, param_info, export_path="pp.pik", install_signal_handlers=False)
    res = posterior_predictive(ms, burn_in=0.5)
    assert res["n_draws"] == 2 * 15
    assert set(res["chains"].tolist()) == {0, 1}
    for m in res["measurements"]:
        lo, med, hi = m["quantiles"]
        assert m["times"].size > 0 and 0 < m["count"].min() and m["count"].max() <= res["n_draws"]
        assert np.all(lo <= med) and np.all(med <= hi)
        assert 0.0 <= m["coverage"] <= 1.0
