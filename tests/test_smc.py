"""CPU tier: the adaptive tempered SMC sampler (metrotrpl_b200.smc) with injected vectorised
likelihoods whose evidence and posterior are known in closed form, its determinism across seeds and
ranks (gloo, world_size 2), its Ensemble, and its refusals."""
import os
import pickle
import sys
import tempfile

import numpy as np
import pytest
from scipy.special import erf
from scipy.stats import truncnorm

from metrotrpl_b200.predictive import posterior_predictive
from metrotrpl_b200.smc import next_beta, smc, systematic_resample
from metrotrpl_b200.trial_move_generation import _approve_rows

NAMES = ["n0", "p0", "mu_n", "mu_p", "ks", "Cn", "Cp", "Sf", "Sb", "tauN", "tauP", "eps", "Tm", "m"]
GUESS = {"n0": 1e8, "p0": 3e15, "mu_n": 20, "mu_p": 20, "ks": 4.8e-11, "Cn": 4.4e-29, "Cp": 4.4e-29,
         "Sf": 10, "Sb": 10, "tauN": 511, "tauP": 871, "eps": 10, "Tm": 300, "m": 1}
LINEAR = ("Tm", "m")
# box (in the parameter's own units) and the Gaussian's centre and width in the sampler's coordinates
# (log10 of the box where do_log is set): every Gaussian sits well inside its box but is cut by it
GAUSS = {"Sf": ((1e-2, 1e3), 0.5, 0.3), "Tm": ((250.0, 350.0), 310.0, 12.0), "Sb": ((1e-1, 1e2), 1.8, 0.4),
         "ks": ((1e-12, 1e-9), -10.2, 0.35), "m": ((0.5, 2.0), 1.1, 0.2)}
SEEDS = range(8)


def problem(active, boxes, tmp=None, **extra):
    """smc()'s positional arguments for the named active parameters and their prior boxes."""
    tmp = tmp or tempfile.mkdtemp()
    t = np.linspace(0, 10, 5)
    sim_info = {"lengths": [300, 300], "nx": [32, 32], "meas_types": ["TRPL", "TRPL"], "num_meas": 2}
    ini = np.ones((2, 32))
    e_data = ([t, t], [np.zeros(5)] * 2, [np.full(5, 0.1)] * 2)
    param_info = {"names": list(NAMES), "active": {n: int(n in active) for n in NAMES},
                  "unit_conversions": {}, "do_log": {n: int(n not in LINEAR) for n in NAMES},
                  "prior_dist": {n: (0, np.inf) for n in NAMES}, "init_guess": dict(GUESS),
                  "trial_move": {n: 0.05 for n in NAMES}}
    param_info["prior_dist"].update(boxes)
    MCMC = {"init_cond_path": "x", "measurement_path": "y", "output_path": tmp, "solver": ("solveivp",),
            "model": "std", "ini_mode": "density", "log_y": 1, "rtol": 1e-6, "atol": None,
            "model_uncertainty": {"TRPL": 0.05}, **extra}
    return sim_info, ini, e_data, MCMC, param_info


def coords(states, names):
    """Sampler coordinates of the named columns of linear states."""
    cols = [NAMES.index(n) for n in names]
    return np.where([n in LINEAR for n in names], states[:, cols], np.log10(states[:, cols]))


def box(name):
    a, b = GAUSS[name][0]
    return (a, b) if name in LINEAR else (np.log10(a), np.log10(b))


def gaussian_factory(names, calls=None):
    mu = np.array([GAUSS[n][1] for n in names])
    s = np.array([GAUSS[n][2] for n in names])

    def factory(ef):
        def loglik(states):
            if calls is not None:
                calls.append(np.array(states))
            return -0.5 * (((coords(states, names) - mu) / s) ** 2).sum(axis=1)
        return loglik
    return factory


def gauss_log_z(names, cut=None):
    """log of (1/V) * integral over the box of exp(-|x - mu|^2 / 2 s^2): a product of erf differences.
    cut: {name: (lo, hi)} narrows the integration range of a coordinate, not the volume V."""
    out = 0.0
    for n in names:
        (a, b), mu, s = box(n), GAUSS[n][1], GAUSS[n][2]
        lo, hi = (cut or {}).get(n, (a, b))
        mass = 0.5 * (erf((hi - mu) / (np.sqrt(2) * s)) - erf((lo - mu) / (np.sqrt(2) * s)))
        out += np.log(s * np.sqrt(2 * np.pi) * mass / (b - a))
    return out


def run(names, seed, n=2000, factory=None, **kw):
    sim_info, ini, e_data, MCMC, param_info = problem(names, {k: GAUSS[k][0] for k in names})
    return smc(sim_info, ini, e_data, MCMC, param_info, n_particles=n, seed=seed,
               evaluator_factory=factory or gaussian_factory(names), **kw)


@pytest.mark.parametrize("names", [("Sf", "Tm"), ("Sf", "Tm", "Sb", "ks", "m")])
def test_gaussian_in_a_box_evidence_and_moments(names):
    want = gauss_log_z(names)
    means, variances = [], []
    for seed in SEEDS:
        # 20 sweeps a stage: with 5, the resampled copies stay correlated and log Z spreads 0.08 nats
        # over the seeds in 5 dimensions (0.025 with 20)
        ms = run(names, seed, n=4000, n_moves=20)
        got = ms.smc["log_evidence"]
        assert abs(got - want) < 0.1, (seed, got, want)
        x = coords(ms.H.states[:, :, 0], names)
        means.append(x.mean(axis=0))
        variances.append(x.var(axis=0))
        assert ms.smc["beta"][-1] == ms.smc["beta"][-2] == 1.0 and np.all(np.diff(ms.smc["beta"]) >= 0)
    means, variances = np.array(means), np.array(variances)
    t_mean, t_var = [], []
    for n in names:
        (a, b), mu, s = box(n), GAUSS[n][1], GAUSS[n][2]
        d = truncnorm((a - mu) / s, (b - mu) / s, loc=mu, scale=s)
        t_mean.append(d.mean())
        t_var.append(d.var())
    # Monte Carlo error of the 8-seed average, from the seeds' spread
    for got, true in ((means, np.array(t_mean)), (variances, np.array(t_var))):
        err = got.std(axis=0, ddof=1) / np.sqrt(len(got))
        assert np.all(np.abs(got.mean(axis=0) - true) <= 4 * err), (got.mean(axis=0), true, err)


def test_two_separated_modes_keep_their_masses():
    names = ("Sf", "Tm")
    s = np.array([0.15, 10.0])
    centres = np.array([[-1.0, 300.0], [2.0, 300.0]])
    weights = np.array([0.25, 0.75])

    def factory(ef):
        def loglik(states):
            x = coords(states, names)
            comp = [-0.5 * (((x - c) / s) ** 2).sum(axis=1) for c in centres]
            return np.logaddexp(np.log(weights[0]) + comp[0], np.log(weights[1]) + comp[1])
        return loglik
    for seed in range(3):
        ms = run(names, seed, n=4000, factory=factory)
        x = coords(ms.H.states[:, :, 0], names)
        frac = np.mean(x[:, 0] < 0.5)
        assert abs(frac - 0.25) <= 0.05, (seed, frac)
        want = np.log(2 * np.pi * s.prod() / (5.0 * 100.0))        # both modes lie well inside the box
        assert abs(ms.smc["log_evidence"] - want) < 0.1


def test_forbidden_region_gives_the_truncated_evidence():
    """L = 0 (as -inf, and as NaN) over 52 % of the box: the evidence is that of the truncated target,
    and the first reweighting (fewer live particles than the ESS target) takes the smallest step."""
    names = ("Sf", "Tm")
    inner = gaussian_factory(names)

    def factory(ef):
        f = inner(ef)

        def loglik(states):
            x = coords(states, names)
            ll = f(states)
            ll[x[:, 0] > 1.0] = -np.inf             # Sf above 10: a failed integration
            ll[x[:, 1] < 270.0] = np.nan            # Tm below 270: NaN
            return ll
        return loglik
    # live share of the box: (1 - (-2)) / 5 * (350 - 270) / 100 = 0.48 < ess_target
    want = gauss_log_z(names, cut={"Sf": (-2.0, 1.0), "Tm": (270.0, 350.0)})
    for seed in range(4):
        ms = run(names, seed, n=4000, factory=factory)
        assert abs(ms.smc["log_evidence"] - want) < 0.1, (seed, ms.smc["log_evidence"], want)
        assert ms.smc["beta"][1] < 1e-300
        x = coords(ms.H.states[:, :, 0], names)
        assert np.all((x[:, 0] <= 1.0) & (x[:, 1] >= 270.0)) and np.all(np.isfinite(ms.H.loglikelihood))


def test_prior_support_and_inactive_parameters():
    """tauN, tauP, n0 and p0 active with boxes the checks cut: every particle drawn from the prior and
    every final one passes _approve_rows, and inactive columns are init_guess exactly."""
    names = ("n0", "p0", "tauN", "tauP")
    boxes = {"n0": (1e12, 1e17), "p0": (1e12, 1e17), "tauN": (1.0, 1e5), "tauP": (1.0, 1e5)}
    calls = []

    def factory(ef):
        def loglik(states):
            calls.append(np.array(states))
            x = coords(states, names)
            return -0.5 * (((x[:, 2] - 2.5) / 0.5) ** 2 + ((x[:, 1] - 15.5) / 0.4) ** 2)
        return loglik
    sim_info, ini, e_data, MCMC, param_info = problem(names, boxes)
    ms = smc(sim_info, ini, e_data, MCMC, param_info, n_particles=1000, seed=5, evaluator_factory=factory)
    ef = ms.ensemble_fields
    do_log = np.asarray(ef["do_log"])
    prior, final = calls[0], ms.H.states[:, :, 0]
    assert len(prior) == 1000 and ms.smc["prior_draws"] > 1000       # the checks rejected some draws
    inactive = [i for i, n in enumerate(NAMES) if n not in names]
    for st in (prior, final, *calls[1:]):
        assert np.all(_approve_rows(np.where(do_log, np.log10(st), st), ef))
        assert np.all(st[:, inactive] == np.array([GUESS[NAMES[i]] for i in inactive])[None, :])
    x = coords(prior, names)
    assert np.all(np.abs(x[:, 2] - x[:, 3]) <= 2) and np.all(x[:, 1] > x[:, 0])


def test_same_seed_same_result_and_record():
    a, b = run(("Sf", "Tm"), 11, n=500), run(("Sf", "Tm"), 11, n=500)
    np.testing.assert_array_equal(a.H.states, b.H.states)
    np.testing.assert_array_equal(a.H.loglikelihood, b.H.loglikelihood)
    assert set(a.smc) == {"log_evidence", "seed", "prior_draws", "beta", "ess", "acceptance", "lam",
                          "launches", "trajectories", "wall_time"}
    for k in a.smc:
        if k != "wall_time":
            np.testing.assert_array_equal(a.smc[k], b.smc[k])
    c = run(("Sf", "Tm"), 12, n=500)
    assert not np.array_equal(a.H.states, c.H.states)
    st = a.smc
    n_stages = len(st["beta"])
    assert all(len(st[k]) == n_stages for k in ("ess", "acceptance", "lam", "launches", "trajectories", "wall_time"))
    assert st["beta"][0] == 0 and st["launches"][0] == 1 and st["trajectories"][0] == 500 * 2
    assert np.all(st["launches"][1:] == 5) and np.all(st["trajectories"][1:] <= 5 * 500 * 2)
    assert np.all(st["ess"][1:-1] >= 0.5 * 500 * (1 - 1e-9)) and np.all((st["acceptance"][1:] > 0) & (st["acceptance"][1:] < 1))
    assert a.latest_iter == 1 and a.H.states.shape == (500, len(NAMES), 1)
    assert len(a.unique_fields) == 500 and all(uf["_T"] == 1 for uf in a.unique_fields)


def test_resampling_and_bisection():
    rng = np.random.default_rng(0)
    w = np.array([0.0, 0.5, 0.0, 0.25, 0.25, 0.0])
    for _ in range(50):
        idx = systematic_resample(rng, w)
        counts = np.bincount(idx, minlength=6)
        assert counts[[0, 2, 5]].sum() == 0 and counts[1] == 3 and counts[3] + counts[4] == 3
    ll = rng.normal(0, 30, 1000)
    beta = next_beta(0.2, ll, 500.0)
    w = np.exp((beta - 0.2) * (ll - ll.max()))
    assert 0.2 < beta < 1 and abs(w.sum() ** 2 / (w ** 2).sum() - 500) < 1e-6
    assert next_beta(0.2, np.zeros(10), 5.0) == 1.0


def test_result_feeds_posterior_predictive_and_pickles():
    from tests.emu import quantiles_emu as emu
    names = ("Sf", "Tm")
    tmp = tempfile.mkdtemp()
    sim_info, ini, e_data, MCMC, param_info = problem(names, {k: GAUSS[k][0] for k in names}, tmp=tmp)
    ms = smc(sim_info, ini, e_data, MCMC, param_info, n_particles=300, seed=2, export_path="smc.pik",
             evaluator_factory=gaussian_factory(names))
    with open(os.path.join(tmp, "smc.pik"), "rb") as f:
        back = pickle.load(f)
    np.testing.assert_array_equal(back.H.states, ms.H.states)
    np.testing.assert_array_equal(back.H.loglikelihood, ms.H.loglikelihood)
    assert back.smc["log_evidence"] == ms.smc["log_evidence"]
    seen = {}

    def evaluator(states):
        seen["states"] = states
        x = coords(states, names)
        fit = np.concatenate([x[:, :1] + 0.1 * np.arange(5)[None, :]] * 2, axis=1)
        return (*emu.fit_quantiles(fit, (0.05, 0.5, 0.95)), np.zeros((len(states), 2), dtype=np.int32))
    res = posterior_predictive(back, quantiles=(0.05, 0.5, 0.95), burn_in=0, evaluator=evaluator)
    assert res["n_draws"] == 300
    np.testing.assert_array_equal(seen["states"], ms.H.states[:, :, 0])
    assert len(res["measurements"]) == 2 and all(0 <= m["coverage"] <= 1 for m in res["measurements"])


def test_bad_inputs_are_refused():
    names = ("Sf", "Tm")

    def never(ef):
        raise AssertionError("built a likelihood despite bad arguments")

    def call(boxes=None, extra=None, **kw):
        sim_info, ini, e_data, MCMC, param_info = problem(names, boxes or {k: GAUSS[k][0] for k in names},
                                                          **(extra or {}))
        kw.setdefault("n_particles", 10)
        return smc(sim_info, ini, e_data, MCMC, param_info, seed=0, evaluator_factory=never, **kw)
    for kw, msg in (({"n_particles": 1}, "n_particles"), ({"ess_target": 0.0}, "ess_target"),
                    ({"ess_target": 1.0}, "ess_target"), ({"ess_target": float("nan")}, "ess_target"),
                    ({"n_moves": 0}, "n_moves"),
                    ({"boxes": {"Sf": (1e-2, np.inf), "Tm": (250, 350)}}, "finite"),
                    ({"boxes": {"Sf": (1e-2, 1e3), "Tm": (-np.inf, 350)}}, "finite"),
                    ({"boxes": {"Sf": (0.0, 1e3), "Tm": (250, 350)}}, "positive lower bound"),
                    ({"boxes": {"Sf": (-1.0, 1e3), "Tm": (250, 350)}}, "positive lower bound"),
                    ({"extra": {"do_mu_constraint": (20, 2)}}, "do_mu_constraint")):
        with pytest.raises(ValueError, match=msg):
            call(**kw)
    with pytest.raises(NotImplementedError, match="log_y"):
        call(extra={"log_y": 0})


def _worker(rank, world, port, q):
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank),
                      MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    from metrotrpl_b200.parallel import Comm
    comm = Comm(backend="gloo")
    sizes = []

    def factory(ef):
        f = gaussian_factory(("Sf", "Tm"))(ef)

        def loglik(states):
            sizes.append(len(states))
            return f(states)
        return loglik
    ms = run(("Sf", "Tm"), 3, n=501, factory=factory, comm=comm)
    smc_rec = {k: v for k, v in ms.smc.items() if k != "wall_time"}
    q.put((rank, ms.H.states, ms.H.loglikelihood, smc_rec, sizes))
    comm.barrier()


def test_two_ranks_equal_one_rank_gloo():
    import torch.multiprocessing as mp
    one = run(("Sf", "Tm"), 3, n=501)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + ((os.getpid() + 250) % 500)
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = [q.get(timeout=600) for _ in range(2)]
    for p in procs:
        p.join(timeout=60)
    assert sorted(g[0] for g in got) == [0, 1]
    for rank, states, ll, rec, sizes in got:
        np.testing.assert_array_equal(states, one.H.states)
        np.testing.assert_array_equal(ll, one.H.loglikelihood)
        for k, v in rec.items():
            np.testing.assert_array_equal(v, one.smc[k])
        assert sizes[0] == (251 if rank == 0 else 250)          # each rank evaluated its own block
