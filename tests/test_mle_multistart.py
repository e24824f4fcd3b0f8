"""CPU tier: many-start maximum likelihood and the covariance of the best fit.

nelder_mead_multi runs K Nelder-Mead searches in one batch; every start must walk SciPy's own path
from where it starts (x and fun bit for bit, nit, nfev and message equal), whatever the other starts
do.  best_fit_covariance is checked on a linear model, where Gauss-Newton is exact, and on the host
lock-step build of the kernel source at a zero-residual optimum, against second differences of the
log-likelihood."""
import tempfile

import numpy as np
import pytest
from scipy import stats
from scipy.optimize import minimize

from metrotrpl_b200 import _capi
from metrotrpl_b200.max_likelihood import (best_fit_covariance, draw_starts, fits_by_measurement, mle,
                                           nelder_mead_batched, nelder_mead_multi)
from metrotrpl_b200.sim_utils import Ensemble
from tests.test_metropolis_batched import GUESS, small_problem

# precision vs second differences of the summed log-likelihood at a zero-residual optimum, relative
# to sqrt(H_ii H_jj); measured 1.2e-5 (host build, rtol 1e-9, second-difference step 1e-3)
HESSIAN_TOL = 1e-4
# |grad| at that optimum relative to max|H| * step; measured 6.5e-6
GRAD_TOL = 1e-4


def rosen(x):
    x = np.asarray(x)
    return float(np.sum(100.0 * (x[1:] - x[:-1] ** 2) ** 2 + (1 - x[:-1]) ** 2))


def two_well(x):
    """Global minimum near x0 = -1, a local one near x0 = +1; the other coordinates are a bowl."""
    x = np.asarray(x)
    return float((x[0] ** 2 - 1) ** 2 + 0.3 * x[0] + np.sum((x[1:] - 0.5) ** 2))


def run_multi(f, X0, **kw):
    """nelder_mead_multi with a per-iteration count of fun_batch calls."""
    calls, per_iter = [0], []

    def fun_batch(X):
        calls[0] += 1
        return [f(x) for x in X]

    def cb(idx, x, fx):
        per_iter.append(calls[0])
        calls[0] = 0
    res = nelder_mead_multi(fun_batch, X0, callback=cb, **kw)
    return res, per_iter


def starts_for(n_dim, k, seed):
    rng = np.random.default_rng(seed)
    X0 = rng.uniform(-2, 2, size=(k, n_dim))
    X0[0] = 0.0                                # the zero-coordinate initial simplex (zdelt)
    return X0


@pytest.mark.parametrize("f,n_dim", [(rosen, 2), (rosen, 4), (two_well, 2), (two_well, 3)],
                         ids=["rosen2", "rosen4", "two_well2", "two_well3"])
@pytest.mark.parametrize("k", [1, 7, 64])
@pytest.mark.parametrize("limits", [{}, {"maxiter": 40}, {"maxfev": 57}, {"maxfev": 3}, {"maxiter": 60, "maxfev": 200}],
                         ids=["default", "maxiter", "maxfev", "maxfev_initial", "both"])
def test_every_start_walks_scipys_path(f, n_dim, k, limits):
    X0 = starts_for(n_dim, k, seed=k * 10 + n_dim)
    res, per_iter = run_multi(f, X0, **limits)
    assert max(per_iter, default=0) <= 2
    for s in range(k):
        ref = minimize(f, X0[s], method="Nelder-Mead", options=limits)
        assert np.array_equal(res["x"][s], ref.x), s
        assert res["fun"][s] == ref.fun, s
        assert (res["nit"][s], res["nfev"][s], res["message"][s]) == (ref.nit, ref.nfev, ref.message), s
    if k == 64 and not limits:
        assert len(set(res["nit"].tolist())) > 10             # starts finish at different iterations
        assert any(n == 2 for n in per_iter)                   # some iterations shrink


def test_limits_are_exercised():
    """The cases above reach each exit, and SciPy's budget runs out mid-iteration (shrinks included)."""
    X0 = starts_for(4, 64, seed=44)
    res, _ = run_multi(rosen, X0, maxfev=57)
    assert all(m.startswith("Maximum number of function evaluations") for m in res["message"])
    assert np.all(res["nfev"] == 57)
    res, _ = run_multi(rosen, X0, maxiter=40)
    assert all(m.startswith("Maximum number of iterations") for m in res["message"])


def test_batch_composition_does_not_change_a_start():
    X0 = starts_for(3, 32, seed=5)
    full, _ = run_multi(two_well, X0)
    perm = np.random.default_rng(1).permutation(32)
    shuffled, _ = run_multi(two_well, X0[perm])
    alone = [nelder_mead_batched(lambda X: [two_well(x) for x in X], X0[s]) for s in range(0, 32, 5)]
    for key in ("x", "fun", "nit", "nfev"):
        np.testing.assert_array_equal(shuffled[key], full[key][perm])
    for s, r in zip(range(0, 32, 5), alone):
        assert np.array_equal(r["x"], full["x"][s]) and r["fun"] == full["fun"][s] and r["nit"] == full["nit"][s]


# --- mle(starts=...) ----------------------------------------------------------------------------

ACT2 = ("Sf", "tauN")          # in the order of param_info["names"]


CENTRE = np.array([0.5, 2.5])


def two_well_problem(tmp):
    """small_problem with two active parameters (Sf, tauN) and a two-well log-likelihood in
    u = log10(state) - CENTRE, the wells along Sf: init_guess sits in the local one."""
    sim_info, ini, e_data, MCMC, param_info = small_problem(tmp, n_chains=1)
    MCMC.pop("parallel_tempering")
    MCMC["current_sigma"] = {"TRPL": 0.05}
    for n in param_info["active"]:
        param_info["active"][n] = int(n in ACT2)
    param_info["prior_dist"].update(tauN=(1.0, 1e5), Sf=(1e-2, 1e3))
    act = [param_info["names"].index(n) for n in ACT2]
    param_info["init_guess"] = dict(param_info["init_guess"], Sf=10 ** 1.6, tauN=10 ** 2.9)

    def fake(states):
        u = np.log10(states[:, act]) - CENTRE
        return -np.array([two_well(v) for v in u])
    return sim_info, ini, e_data, MCMC, param_info, act, fake


def scipy_chain(fake, act, base, x0):
    """SciPy's Nelder-Mead on the same cost, with the best vertex after every iteration."""
    path = []

    def cost(x):
        st = base.copy()
        st[act] = 10 ** x
        ll = float(fake(st[None, :])[0])
        return -ll if np.isfinite(ll) else np.inf
    def cb(intermediate_result):
        path.append((intermediate_result.x.copy(), intermediate_result.fun))
    ref = minimize(cost, x0, method="Nelder-Mead", callback=cb)
    return ref, path


def test_mle_single_start_is_scipys_search():
    sim_info, ini, e_data, MCMC, param_info, act, fake = two_well_problem(tempfile.mkdtemp())
    base = np.array([param_info["init_guess"][n] for n in param_info["names"]], dtype=float)
    ms = mle(e_data, sim_info, param_info, ini, MCMC, "mle.pik", None, evaluator=fake)
    ref, path = scipy_chain(fake, act, base, np.log10(base[act]))
    assert set(ms.opt) == {"x", "fun", "nit", "nfev", "nbatch", "npoints", "message"}
    assert np.array_equal(ms.opt["x"], ref.x) and ms.opt["fun"] == ref.fun
    assert (ms.opt["nit"], ms.opt["nfev"], ms.opt["message"]) == (ref.nit, ref.nfev, ref.message)
    assert ms.H.states.shape[2] == len(path) + 1
    np.testing.assert_array_equal(ms.H.states[0, :, 0], base)
    np.testing.assert_array_equal(ms.H.states[0, act, 1:], 10 ** np.array([p[0] for p in path]).T)
    np.testing.assert_array_equal(ms.H.loglikelihood[0, 1:], -np.array([p[1] for p in path]))


def test_mle_many_starts_finds_the_global_well():
    tmp = tempfile.mkdtemp()
    sim_info, ini, e_data, MCMC, param_info, act, fake = two_well_problem(tmp)
    single = mle(e_data, sim_info, param_info, ini, MCMC, None, None, evaluator=fake)
    sim_info, ini, e_data, MCMC, param_info, act, fake = two_well_problem(tmp)
    multi = mle(e_data, sim_info, param_info, ini, MCMC, "mle.pik", None, evaluator=fake, starts=12, seed=3)
    st = multi.opt["starts"]
    assert len(st["fun"]) == 12 and st["message"][0] == single.opt["message"]
    # start 0 is init_guess and reproduces the single-start search
    assert np.array_equal(st["x"][0], single.opt["x"]) and st["fun"][0] == single.opt["fun"]
    assert (st["nit"][0], st["nfev"][0]) == (single.opt["nit"], single.opt["nfev"])
    # ... which stays in the local well; the best start reaches the global one
    assert single.opt["x"][0] - CENTRE[0] > 0.5
    b = multi.opt["best_start"]
    assert b != 0 and multi.opt["x"][0] - CENTRE[0] < -0.5
    assert multi.opt["fun"] == st["fun"].min() < single.opt["fun"]
    # the chain is the best start's: from its start state to its best vertex
    np.testing.assert_array_equal(np.log10(multi.H.states[0, act, 0]), st["x0"][b])
    np.testing.assert_array_equal(multi.H.states[0, act, -1], 10 ** multi.opt["x"])
    assert multi.H.states.shape[2] == multi.opt["nit"]
    ref, path = scipy_chain(fake, act, single.H.states[0, :, 0], st["x0"][b])
    np.testing.assert_array_equal(multi.H.loglikelihood[0, 1:], -np.array([p[1] for p in path]))


def test_mle_explicit_start_array():
    sim_info, ini, e_data, MCMC, param_info, act, fake = two_well_problem(tempfile.mkdtemp())
    base = np.array([param_info["init_guess"][n] for n in param_info["names"]], dtype=float)
    arr = np.repeat(base[None, :], 3, axis=0)
    arr[:, act] = [[10 ** 1.6, 10 ** 2.9], [10 ** -0.4, 10 ** 2.2], [10 ** 1.1, 10 ** 2.0]]
    arr[1, 0] *= 7                                 # an inactive column: held at init_guess
    ms = mle(e_data, sim_info, param_info, ini, MCMC, None, None, evaluator=fake, starts=arr)
    np.testing.assert_array_equal(ms.opt["starts"]["x0"], np.log10(arr[:, act]))
    b = ms.opt["best_start"]
    np.testing.assert_array_equal(ms.H.states[0, 0, :], base[0])


def test_draw_starts():
    sim_info, ini, e_data, MCMC, param_info = small_problem(tempfile.mkdtemp(), n_chains=1)
    param_info["prior_dist"].update(tauN=(1.0, 1e4), Sf=(1e-2, 1e3), p0=(1e14, 1e16), ks=(1e-12, 1e-9),
                                    tauP=(100.0, 900.0))
    param_info["do_log"]["tauP"] = 0
    ens = Ensemble(param_info, sim_info, MCMC, 2)
    ef = ens.ensemble_fields
    state = ens.H.states[0, :, 0]
    a = draw_starts(ef, state, 4001, seed=11)
    np.testing.assert_array_equal(a, draw_starts(ef, state, 4001, seed=11))
    assert not np.array_equal(a, draw_starts(ef, state, 4001, seed=12))
    np.testing.assert_array_equal(a[0], state)
    np.testing.assert_array_equal(a[:, ~ef["active"]], np.repeat(state[None, ~ef["active"]], 4001, axis=0))
    for i in np.flatnonzero(ef["active"]):
        lo, hi = ef["prior_dist"][ef["names"][i]]
        col = a[1:, i]
        assert np.all((col >= lo) & (col <= hi))
        if ef["do_log"][i]:
            u = (np.log10(col) - np.log10(lo)) / (np.log10(hi) - np.log10(lo))
        else:
            u = (col - lo) / (hi - lo)
        assert stats.kstest(u, "uniform").pvalue > 1e-3, ef["names"][i]
    # the global generator is neither used nor disturbed
    np.random.seed(0)
    before = np.random.random()
    np.random.seed(0)
    draw_starts(ef, state, 10, seed=1)
    assert np.random.random() == before
    ef["prior_dist"]["tauN"] = (0, np.inf)
    with pytest.raises(ValueError, match="tauN"):
        draw_starts(ef, state, 3, seed=1)


# --- best_fit_covariance --------------------------------------------------------------------------

def ensemble_at(state_by_name, active, tmp):
    """An Ensemble whose chain is the one state given (what best_fit_covariance reads)."""
    sim_info, ini, e_data, MCMC, param_info = small_problem(tmp, n_chains=1)
    MCMC.pop("parallel_tempering")
    MCMC["current_sigma"] = {"TRPL": 0.05}
    for n in param_info["active"]:
        param_info["active"][n] = int(n in active)
    param_info["init_guess"] = dict(param_info["init_guess"], **state_by_name)
    return Ensemble(param_info, sim_info, MCMC, 1), sim_info, ini, e_data


def test_covariance_of_a_linear_model():
    act_names = ("p0", "ks", "Sf", "tauN")
    ens, *_ = ensemble_at({}, act_names, tempfile.mkdtemp())
    ef = ens.ensemble_fields
    act = ef["active"]
    rng = np.random.default_rng(4)
    A = [rng.normal(size=(9, 4)), rng.normal(size=(7, 4))]
    v = [rng.normal(size=9), rng.normal(size=7)]
    u = [rng.uniform(0.01, 0.1, 9), rng.uniform(0.01, 0.1, 7)]
    sig = [0.05, 0.2]
    n_c = [9, 5]                                   # measurement 1 compares a prefix of 5 points

    def linear(states):
        x = np.log10(states[:, act])
        fits = []
        for m in range(2):
            f = x @ A[m].T
            f[:, n_c[m]:] = np.nan
            fits.append(f)
        return fits, v, u, sig

    out = best_fit_covariance(ens, evaluator=linear)
    assert out["ok"] and out["names"] == list(act_names)
    W = [1 / (sig[m] ** 2 + 2 * u[m][:n_c[m]] ** 2) for m in range(2)]
    prec = sum(2 * A[m][:n_c[m]].T @ np.diag(W[m]) @ A[m][:n_c[m]] for m in range(2))
    cov = np.linalg.inv(prec)
    np.testing.assert_allclose(out["precision"], prec, rtol=1e-10, atol=0)
    np.testing.assert_allclose(out["cov"], cov, rtol=1e-10, atol=1e-10 * np.abs(cov).max())
    np.testing.assert_allclose(out["std"], np.sqrt(np.diag(cov)), rtol=1e-10)
    np.testing.assert_allclose(np.diag(out["corr"]), 1.0, rtol=1e-12)
    x = out["x"]
    grad = -sum(2 * A[m][:n_c[m]].T @ (W[m] * (A[m][:n_c[m]] @ x - v[m][:n_c[m]])) for m in range(2))
    np.testing.assert_allclose(out["grad"], grad, rtol=1e-6)
    # a compared prefix that changes with the state is refused
    def shifting(states):
        fits, *rest = linear(states)
        fits[0][1, 8] = np.nan
        return (fits, *rest)
    bad = best_fit_covariance(ens, evaluator=shifting)
    assert not bad["ok"] and "change" in bad["reason"] and np.all(np.isnan(bad["cov"]))


def host_problem(tmp, act_names, theta=None, max_steps=_capi.DEFAULT_MAX_STEPS):
    """small_problem whose data are the host build's own fitted curves at theta: a zero-residual
    optimum.  Returns (ensemble at theta, evaluator of the host build, log-likelihood of states)."""
    from tests.emu import emu
    ens, sim_info, ini, e_data = ensemble_at(theta or {}, act_names, tmp)
    ef = ens.ensemble_fields
    idx, units = ef["_param_indexes"], ef["units"]
    t, _, uncs = e_data
    prob = _capi.pack_problem(sim_info, ini, t, e_data[1], uncs)
    opts = _capi.make_opts(RTOL=1e-9, max_steps=max_steps)
    star = ens.H.states[0, :, 0]

    def run(prob, states):
        params = _capi.pack_params(states, idx, units)
        aux = _capi.default_aux(len(states), 2, [0.05, 0.05])
        return emu.loglik_batch(prob, params, aux, opts, want_curves=False, fit=True)

    fit0 = run(prob, star[None, :])[4][0]
    vals = [fit0[:len(t[0])], fit0[len(t[0]):]]
    prob = _capi.pack_problem(sim_info, ini, t, vals, uncs)

    def evaluator(states):
        ll, st, _, _, fit = run(prob, states)
        return (*fits_by_measurement(prob, fit, st, ll), [0.05, 0.05])

    def loglik(states):
        return run(prob, states)[0][:, :, 0].sum(axis=1)
    return ens, evaluator, loglik


def second_differences(loglik, state, active, h):
    """Hessian of -loglik in log10 of the active parameters by second differences."""
    x = np.log10(state[active])
    P = len(x)
    pts = [np.zeros(P)]
    for i in range(P):
        for j in range(i, P):
            for si, sj in ((1, 1), (1, -1), (-1, 1), (-1, -1)):
                d = np.zeros(P)
                d[i] += si * h
                d[j] += sj * h
                pts.append(d)
    states = np.repeat(state[None, :], len(pts), axis=0)
    states[:, active] = 10 ** (x + np.array(pts))
    states[0] = state
    ll = loglik(states)
    H = np.zeros((P, P))
    k = 1
    for i in range(P):
        for j in range(i, P):
            pp, pm, mp, mm = ll[k:k + 4]
            k += 4
            H[i, j] = H[j, i] = -(pp - pm - mp + mm) / (4 * h * h)
    return H


def test_covariance_on_the_host_build_matches_the_hessian():
    ens, evaluator, loglik = host_problem(tempfile.mkdtemp(), ("p0", "ks", "Sf", "tauN"))
    out = best_fit_covariance(ens, evaluator=evaluator)
    assert out["ok"], out["reason"]
    ef = ens.ensemble_fields
    H_fd = second_differences(loglik, ens.H.states[0, :, -1], ef["active"], 1e-3)
    scale = np.sqrt(np.outer(np.diag(out["precision"]), np.diag(out["precision"])))
    err = np.abs(H_fd - out["precision"]) / scale
    print(f"precision vs second differences: {err.max():.2e}; "
          f"|grad| / (max|H| step): {np.abs(out['grad']).max() / (np.abs(out['precision']).max() * 1e-4):.2e}")
    assert err.max() <= HESSIAN_TOL
    assert np.abs(out["grad"]).max() <= GRAD_TOL * np.abs(out["precision"]).max() * 1e-4
    assert np.all(np.isfinite(out["std"])) and np.all(np.abs(out["corr"]) <= 1 + 1e-12)


def test_covariance_refuses_an_unidentifiable_parameter():
    # 'm' does not enter the 'std' model: its column of the Jacobian is zero
    ens, evaluator, _ = host_problem(tempfile.mkdtemp(), ("ks", "tauN", "m"))
    out = best_fit_covariance(ens, evaluator=evaluator)
    assert not out["ok"] and "positive definite" in out["reason"]
    assert np.all(np.isnan(out["cov"])) and np.all(np.isnan(out["std"]))
    assert np.all(out["precision"][2] == 0)


def test_covariance_refuses_a_failed_evaluation():
    # a step budget too small for the curves: TRPL_ST_MAX_STEPS on every trajectory
    ens, evaluator, _ = host_problem(tempfile.mkdtemp(), ("ks", "tauN"))
    _, failing, _ = host_problem(tempfile.mkdtemp(), ("ks", "tauN"), max_steps=3)
    assert best_fit_covariance(ens, evaluator=evaluator)["ok"]
    out = best_fit_covariance(ens, evaluator=failing)
    assert not out["ok"] and "evaluation failed" in out["reason"]
    assert np.all(np.isnan(out["cov"]))
