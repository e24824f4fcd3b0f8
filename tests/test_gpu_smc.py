"""GPU tier: adaptive tempered SMC through the CUDA likelihood on the six-curve staub problem, with
tauN and Sf active (the fixture the many-start MLE tests fit).

The reference value is a tensor-grid quadrature of the same CUDA likelihood (smc.make_cuda_loglik)
over the prior's support: log Z = log((1 / V) * integral of L), V the support's area in (log10 tauN,
log10 Sf).  The posterior is far narrower than the box, so the grid covers a sub-box around it, and
the test shows that the sub-box holds the mass: L on its edge, and on a coarse grid over the rest of
the box, is below max L by more than EDGE_NATS.  Where the posterior reaches the prior box's own
boundary (small Sf: the surface then recombines nothing the data can see), the sub-box extends to it.  The model uncertainty is the fixture's own; the
posterior is resolved on the sub-box grid without widening it.
"""
import tempfile

import numpy as np
import pytest

from metrotrpl_b200.predictive import posterior_predictive
from metrotrpl_b200.smc import make_cuda_loglik, prior_box, smc
from metrotrpl_b200.trial_move_generation import _approve_rows
from tests.test_gpu_mle_multistart import staub_mle_inputs

pytestmark = pytest.mark.gpu

N = 4096
MOVES = 10
SEEDS = (0, 1, 2, 3)
EDGE_NATS = 20.0            # L outside the integration sub-box is below max L by at least this much
GRID = 128                  # cells per axis of the sub-box; GRID / 2 shows the quadrature is resolved
QUANTILES = (0.05, 0.5, 0.95)


def run(seed):
    e_data, sim_info, param_info, ini, MCMC = staub_mle_inputs(tempfile.mkdtemp())
    return smc(sim_info, ini, e_data, MCMC, param_info, n_particles=N, n_moves=MOVES, seed=seed)


def active_coords(ms):
    ef = ms.ensemble_fields
    return np.log10(ms.H.states[:, ef["active"], 0])            # both parameters are do_log


@pytest.fixture(scope="module")
def runs():
    return [run(s) for s in SEEDS]


@pytest.fixture(scope="module")
def quadrature(runs):
    ms = runs[0]
    ef = ms.ensemble_fields
    active = ef["active"]
    lo, hi = prior_box(ef)
    loglik = make_cuda_loglik(ef, ms.unique_fields[0]["current_sigma"])
    base = ms.H.states[0, :, 0].copy()
    do_log = ef["do_log"]

    def ll_at(x):
        states = np.repeat(base[None, :], len(x), axis=0)
        states[:, active] = 10 ** x
        full = np.where(do_log, np.log10(states), states)
        assert np.all(_approve_rows(full, ef))                  # the checks do not cut this box
        return loglik(states)

    def grid(a, b, n):
        """Cell centres of an n x n grid on [a, b], as [n * n, 2], and the cell area."""
        c = [a[i] + (np.arange(n) + 0.5) * (b[i] - a[i]) / n for i in range(2)]
        g = np.stack(np.meshgrid(*c, indexing="ij"), axis=-1).reshape(-1, 2)
        return g, c, np.prod((b - a) / n)

    # the sub-box: the particles' range of every seed, widened by all of it on each side, inside the box
    x = np.concatenate([active_coords(r) for r in runs])
    span = x.max(axis=0) - x.min(axis=0)
    a = np.maximum(lo, x.min(axis=0) - span)
    b = np.minimum(hi, x.max(axis=0) + span)
    out = {}
    for n in (GRID // 2, GRID):
        g, c, area = grid(a, b, n)
        ll = ll_at(g)
        m = ll.max()
        out[n] = {"log_z": m + np.log(np.exp(ll - m).sum() * area) - np.log(np.prod(hi - lo)),
                  "ll": ll.reshape(n, n), "centres": c, "max": m}
    fine = out[GRID]
    ll = fine["ll"]
    # the sub-box's sides inside the prior box (a side on the prior box's own boundary cuts no mass)
    sides = [(ll[0], a[0] > lo[0]), (ll[-1], b[0] < hi[0]), (ll[:, 0], a[1] > lo[1]), (ll[:, -1], b[1] < hi[1])]
    edge = np.concatenate([v for v, inner in sides if inner] + [[-np.inf]])
    assert edge.max() < fine["max"] - EDGE_NATS, (edge.max(), fine["max"])
    g, _, _ = grid(lo, hi, 96)
    outside = ~np.all((g >= a) & (g <= b), axis=1)
    coarse = ll_at(g[outside])
    assert coarse.max() < fine["max"] - EDGE_NATS, (coarse.max(), fine["max"])
    fine["resolved"] = abs(out[GRID]["log_z"] - out[GRID // 2]["log_z"])
    print(f"quadrature on [{a}, {b}] of the box [{lo}, {hi}]: log Z {out[GRID]['log_z']:.6f} ({GRID}^2), "
          f"{out[GRID // 2]['log_z']:.6f} ({GRID // 2}^2); max log L {fine['max']:.4f}, edge {edge.max():.1f}, "
          f"outside {coarse.max():.1f}")
    return fine


def test_quadrature_is_resolved(quadrature):
    assert quadrature["resolved"] < 0.01


def test_evidence_agrees_with_quadrature(runs, quadrature):
    lz = np.array([r.smc["log_evidence"] for r in runs])
    tol = max(0.1, 4 * lz.std(ddof=1))
    for r in runs:
        st = r.smc
        print(f"seed {st['seed']}: log Z {st['log_evidence']:.4f}, {len(st['beta'])} stages, "
              f"{st['launches'].sum()} launches, {st['trajectories'].sum()} trajectories, "
              f"{st['wall_time'].sum():.2f} s, acceptance {np.round(st['acceptance'][1:], 2)}")
    print(f"quadrature {quadrature['log_z']:.4f}; tolerance {tol:.3f}")
    assert np.all(np.abs(lz - quadrature["log_z"]) <= tol), (lz, quadrature["log_z"])


def test_marginal_quantiles_agree_with_the_grid(runs, quadrature):
    ll = quadrature["ll"]
    p = np.exp(ll - ll.max())
    p /= p.sum()
    q = np.array(QUANTILES)
    for axis in range(2):
        c = quadrature["centres"][axis]
        h = c[1] - c[0]
        marg = p.sum(axis=1 - axis)
        edges = np.concatenate([[c[0] - h / 2], c + h / 2])
        cdf = np.concatenate([[0.0], np.cumsum(marg)])
        want = np.interp(q, cdf, edges)
        dens = np.interp(want, c, marg / h)
        got = np.array([np.quantile(active_coords(r)[:, axis], q) for r in runs])
        # Monte Carlo error of the seeds' average: their spread, or sqrt(q (1 - q) / N) / density per
        # seed with N / 4 independent particles, whichever is larger; plus one grid cell
        err = np.maximum(got.std(axis=0, ddof=1), np.sqrt(q * (1 - q) / (N / 4)) / dens) / np.sqrt(len(runs))
        print(f"axis {axis}: particles {got.mean(axis=0)}, grid {want}, error {err}")
        assert np.all(np.abs(got.mean(axis=0) - want) <= 4 * err + h), (axis, got.mean(axis=0), want, err)


def test_same_seed_is_bit_identical(runs):
    again = run(SEEDS[0])
    np.testing.assert_array_equal(again.H.states, runs[0].H.states)
    np.testing.assert_array_equal(again.H.loglikelihood, runs[0].H.loglikelihood)
    assert again.smc["log_evidence"] == runs[0].smc["log_evidence"]
    for k in ("beta", "ess", "acceptance", "lam", "launches", "trajectories"):
        np.testing.assert_array_equal(again.smc[k], runs[0].smc[k])


def test_posterior_predictive_of_the_particles(runs):
    res = posterior_predictive(runs[0], burn_in=0)
    assert res["n_draws"] == N and res["n_failed"] == 0
    cov = [m["coverage"] for m in res["measurements"]]
    print(f"coverage of the 95 % band per curve: {np.round(cov, 3)}")
    assert len(cov) == 6 and all(0 <= c <= 1 for c in cov)
