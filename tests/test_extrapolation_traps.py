"""CPU tier: the order-6 extrapolation integrator (csrc/extrapolation.h) on the trap-assisted model
at nx = 128, the grid its cooperative kernel serves, and the rule that decides which problems may use
it.  The host lock-step build runs the one-warp driver, whose bits the cooperative kernel reproduces
(test_gpu_extrapolation_traps.py)."""
import os

import numpy as np
import pytest

from metrotrpl_b200 import _capi
from tests.emu import emu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def traps128_problem(irf=True):
    """The traps + IRF problem of tests/golden/traps_irf.npz (configs[3]) on 128 nodes: fluence mode,
    so the initial condition follows the grid.  Returns (fixture, names, idx, prob)."""
    g = np.load(os.path.join(GOLDEN, "traps_irf.npz"))
    names = [str(n) for n in g["names"]]
    idx = {n: i for i, n in enumerate(names)}
    sim = {"lengths": list(g["lengths"]), "nx": [128] * 2, "meas_types": ["TRPL"] * 2, "num_meas": 2}
    kw = dict(irf_convolution=[520, 520], irf_tables={520: (g["moments"], g["t_irf"])}) if irf else {}
    prob = _capi.pack_problem(sim, g["inis"], [g["t"]] * 2, list(g["vals"]), list(g["uncs"]), model="traps",
                              ini_mode="fluence", **kw)
    return g, names, idx, prob


def jittered_states(g, names, n_sets, seed):
    """n_sets fixture states, every parameter but n0, eps, Tm jittered +-0.1 decade (as bench.py
    builds configs[3])."""
    idx = {n: i for i, n in enumerate(names)}
    rng = np.random.default_rng(seed)
    base = g["states"][rng.integers(0, len(g["states"]), n_sets)]
    jit = np.ones_like(base)
    act = [idx[n] for n in names if n not in ("n0", "eps", "Tm", "m")]
    jit[:, act] = 10 ** rng.uniform(-0.1, 0.1, size=(n_sets, len(act)))
    return base * jit


def compare_with_truth(run, truth, rodas, n_t):
    """(max curve error within 12 decades of each curve's start, max relative log-likelihood error,
    mean steps / RODAS4's mean steps) of `run` against `truth`; each a (logll, status, nsteps, curves)
    tuple of the same sets."""
    X = run[3].reshape(-1, 2, n_t)
    T = truth[3].reshape(-1, 2, n_t)
    in_range = T >= 1e-12 * T[:, :, :1]
    curve = float(np.where(in_range, np.abs(X / T - 1), 0.0).max())
    ll = float(np.abs(run[0][:, :, 0] / truth[0][:, :, 0] - 1).max())
    ratio = float(run[2][..., 0].mean() / rodas[2][..., 0].mean())
    return curve, ll, ratio


def test_extrapolation_integrator_traps_irf_on_128_nodes():
    """One-warp driver, traps + IRF at nx = 128, rtol 1e-7, against RODAS4 at rtol 1e-10 in the same
    build (measured: curves 1.7e-6, log-likelihoods 2.9e-7, 0.40x RODAS4's steps)."""
    g, names, idx, prob = traps128_problem()
    params = _capi.pack_params(g["states"], idx, g["units"], model="traps")
    aux = _capi.default_aux(len(params), 2, [1.0] * 2)
    seulex = emu.loglik_batch(prob, params, aux, _capi.make_opts(RTOL=1e-7, flags=_capi.OPT_EXTRAPOLATION), True)
    rodas = emu.loglik_batch(prob, params, aux, _capi.make_opts(RTOL=1e-7), True)
    truth = emu.loglik_batch(prob, params, aux, _capi.make_opts(RTOL=1e-10), True)
    curve, ll, ratio = compare_with_truth(seulex, truth, rodas, len(g["t"]))
    print("curve", curve, "logll", ll, "step ratio", ratio)
    assert curve <= 5e-6
    assert ll <= 1e-6
    assert ratio < 0.5
    assert not np.any(seulex[1] & 7)


def test_extrapolation_eligibility_rule():
    """One rule for PathCache(kernel="seulex") and metro(kernel="seulex"): 'std' or 'traps', nx = 128
    on every measurement."""
    _capi.check_extrapolation_problem("std", [128] * 6)
    _capi.check_extrapolation_problem("traps", [128, 128])
    for model, nx in (("std", [64] * 6), ("traps", [256, 256]), ("traps", [128, 100]), ("std", [128, 129])):
        with pytest.raises(ValueError, match="nx = 128"):
            _capi.check_extrapolation_problem(model, nx)
    with pytest.raises(ValueError, match="nx = 128"):
        _capi.check_extrapolation_problem("other", [128])
