"""GPU tier: every node count the kernels dispatch on, through the C ABI (tests/grid_cases.py), and the
four-warp team (nx 257..512) held to what the two-warp team's tests hold: run-to-run and permutation
determinism at full size, the tempering ladder, queue order and force_min_y, the step-log flush, and
the min_y floor met in the upper half of its 128 lanes."""
import os

import numpy as np
import pytest

from metrotrpl_b200 import _capi
from oracle import trpl_oracle as orc
from tests import grid_cases as gc
from tests.emu import emu

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def ctx():
    c = _capi.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def refs():
    return gc.References()


def make_backend(ctx):
    def backend(prob, params, aux, opts, want_curves):
        ctx.set_problem(prob)
        return ctx.loglik_batch(params, aux, opts, want_curves=want_curves)
    return backend


def host(prob, params, aux, opts, want_curves):
    return emu.loglik_batch(prob, params, aux, opts, want_curves)


def test_every_node_count_and_seam_against_lsoda(ctx, refs):
    worst = gc.check_node_count_seams(make_backend(ctx), refs, host=host)
    for k in sorted(worst):
        print(k, f"{worst[k]:.2e}")


def test_reversed_profile_with_swapped_contacts(ctx):
    print(gc.check_reversal_with_swapped_contacts(make_backend(ctx)))


def test_small_grids_inside_larger_kernels(ctx, refs):
    print(gc.check_mixed_grids(make_backend(ctx), refs, host=host, fma_contracted=True))


def test_grids_the_library_refuses(ctx):
    assert gc.check_grid_refusals(make_backend(ctx))


def _traps_irf_problem(nx):
    """configs[3] (traps + IRF, fluence mode) on a grid of nx nodes."""
    g = np.load(os.path.join(GOLDEN, "traps_irf.npz"))
    names = [str(n) for n in g["names"]]
    idx = {n: i for i, n in enumerate(names)}
    sim = {"lengths": list(g["lengths"]), "nx": [nx] * 2, "meas_types": ["TRPL"] * 2, "num_meas": 2}
    prob = _capi.pack_problem(sim, g["inis"], [g["t"]] * 2, list(g["vals"]), list(g["uncs"]), model="traps",
                              ini_mode="fluence", irf_convolution=[520, 520],
                              irf_tables={520: (g["moments"], g["t_irf"])})
    return g, names, idx, prob


def test_four_warp_team_is_deterministic_at_full_size(ctx):
    """1024 jittered parameter sets x 2 curves (traps + IRF, nx = 512) through the four-warp team:
    a second launch reproduces the first bit for bit, a permuted launch permutes the results bit for
    bit (whichever team and SM a trajectory gets, however its four warps meet at the three mailbox
    boundaries), and a sample agrees with the host lock-step build of the same source."""
    g, names, idx, prob = _traps_irf_problem(512)
    n_sets = 1024
    rng = np.random.default_rng(11)
    base = g["states"][rng.integers(0, len(g["states"]), n_sets)]
    jit = np.ones_like(base)
    act = [idx[n] for n in names if n not in ("n0", "eps", "Tm", "m")]
    jit[:, act] = 10 ** rng.uniform(-0.1, 0.1, size=(n_sets, len(act)))
    params = _capi.pack_params(base * jit, idx, g["units"], model="traps")
    aux = _capi.default_aux(n_sets, 2, [1.0] * 2)
    opts = _capi.make_opts(RTOL=1e-7)
    ctx.set_problem(prob)
    ll_a, st_a, ns_a, cur_a = ctx.loglik_batch(params, aux, opts, want_curves=True)
    ll_b, st_b, ns_b, cur_b = ctx.loglik_batch(params, aux, opts, want_curves=True)
    np.testing.assert_array_equal(ll_a, ll_b)
    np.testing.assert_array_equal(ns_a, ns_b)
    np.testing.assert_array_equal(st_a, st_b)
    np.testing.assert_array_equal(cur_a, cur_b)
    perm = rng.permutation(n_sets)
    ll_p, st_p, ns_p, cur_p = ctx.loglik_batch(params[perm], aux[perm], opts, want_curves=True)
    np.testing.assert_array_equal(ll_p, ll_a[perm])
    np.testing.assert_array_equal(ns_p, ns_a[perm])
    np.testing.assert_array_equal(st_p, st_a[perm])
    np.testing.assert_array_equal(cur_p, cur_a[perm])
    assert np.all(np.isfinite(ll_a[..., 0])) and not np.any(st_a & 7)
    sel = np.arange(0, n_sets, 128)
    ll_e, st_e, ns_e, _ = emu.loglik_batch(prob, params[sel], aux[sel], opts, True)
    np.testing.assert_allclose(ll_a[sel], ll_e, rtol=1e-6)
    assert np.abs(ns_a[sel][..., 0] - ns_e[..., 0]).max() <= 5


@pytest.mark.parametrize("nx", [400, 512])
def test_four_warp_team_ladder_queue_order_and_min_y_floor(ctx, nx):
    """The options of the one-warp path through the four-warp team (traps + IRF), padded (400) and
    padding-free (512): the tempering ladder equals the three temperature slots of a plain call, the
    per-chain ladder rows are their sums over the curves, an explicit queue order changes nothing, and
    force_min_y is the host lock-step build's to rounding."""
    g, names, idx, prob = _traps_irf_problem(nx)
    params = _capi.pack_params(g["states"], idx, g["units"], model="traps")
    n = params.shape[0]
    ctx.set_problem(prob)
    opts = _capi.make_opts(RTOL=1e-7)
    aux = _capi.default_aux(n, 2, [1.0] * 2, temps=(1.0, 2.0, 8.0))
    ll, st, ns, cur = ctx.loglik_batch(params, aux, opts, want_curves=True)
    assert not np.any(st & 7)
    ctx.set_ladder(np.array([1.0, 2.0, 8.0, 64.0]))
    aux1 = _capi.default_aux(n, 2, [1.0] * 2, temps=(1.0, 1.0, 1.0))
    ctx.loglik_batch(params, aux1, _capi.make_opts(RTOL=1e-7, flags=_capi.OPT_LADDER), want_curves=False)
    lad = ctx.download_ladder(n)
    np.testing.assert_allclose(lad[:, :, :3], ll, rtol=1e-12)
    assert np.all(lad[:, :, 3] > lad[:, :, 2])
    rows, _ = ctx.download_ladder_sums(n)
    np.testing.assert_allclose(rows, lad.sum(axis=1), rtol=1e-14)
    ctx.set_queue_order(np.random.default_rng(0).permutation(2 * n))
    ll_p, st_p, ns_p, cur_p = ctx.loglik_batch(params, aux, opts, want_curves=True)
    ctx.set_queue_order(None)
    np.testing.assert_array_equal(ll_p, ll)
    np.testing.assert_array_equal(cur_p, cur)
    np.testing.assert_array_equal(ns_p, ns)
    o_f = _capi.make_opts(RTOL=1e-7, flags=_capi.OPT_FORCE_MIN_Y)
    ll_f, _, _, _ = ctx.loglik_batch(params, aux, o_f, want_curves=True)
    ll_e, _, _, _ = emu.loglik_batch(prob, params, aux, o_f, True)
    np.testing.assert_allclose(ll_f, ll_e, rtol=1e-6)


def test_step_log_flush_in_the_four_warp_team_kernel(ctx):
    """A 0.04 ns step cap at nx = 512 (traps + IRF) forces more than 2048 steps per curve: the
    1024-entry step log is flushed at least twice mid-run, 128 measurement times per emission.  Same
    curves and likelihoods as the uncapped run."""
    g, names, idx, prob = _traps_irf_problem(512)
    params = _capi.pack_params(g["states"][:2], idx, g["units"], model="traps")
    aux = _capi.default_aux(2, 2, [1.0] * 2)
    ctx.set_problem(prob)
    free = ctx.loglik_batch(params, aux, _capi.make_opts(RTOL=1e-7), want_curves=True)
    capped = ctx.loglik_batch(params, aux, _capi.make_opts(RTOL=1e-7, hmax=0.04, honor_hmax=True), want_curves=True)
    print("steps free", free[2][..., 0].tolist(), "capped", capped[2][..., 0].tolist())
    assert capped[2][..., 0].min() > 2100 and free[2][..., 0].max() < 1024
    np.testing.assert_allclose(capped[3], free[3], rtol=3e-5)
    np.testing.assert_allclose(capped[0], free[0], rtol=2e-6)
    assert not np.any(capped[1] & 7)


def test_min_y_floor_first_met_in_the_upper_lanes_of_an_emission(ctx):
    """The emission evaluates 128 measurement times per pass on the four-warp team, and the floor
    (forward_solver.py:190-192: from the first value below min_y on, the curve IS min_y) is found by a
    128-bit ballot.  Two curves on 481 times (nx = 512) whose floors are first met at points 100 and
    228, i.e. lanes 100 and 100 of the first and second 128-wide pass, in the upper 64 bits of the
    ballot: the curves before those points are the unfloored ones, from there on exactly min_y, as on
    the host lock-step build and in the oracle."""
    nx, t = 512, np.linspace(0, 60, 481)
    firsts = (100, 228)
    params = gc.params_of("std", [gc.state_of("std", "stiff")])
    aux = _capi.default_aux(1, 2, [gc.SIGMA] * 2)
    opts = _capi.make_opts(RTOL=gc.RTOL)
    free_prob = gc.pack([nx, nx], ["TRPL", "TRPL"], times=t)
    ctx.set_problem(free_prob)
    free = gc.split(free_prob, ctx.loglik_batch(params, aux, opts, want_curves=True)[3][0])
    assert all(np.all(np.diff(c) < 0) for c in free)
    min_y = [float(np.sqrt(c[k - 1] * c[k])) for c, k in zip(free, firsts)]
    prob = gc.pack([nx, nx], ["TRPL", "TRPL"], times=t, min_y=min_y)
    ll, st, ns, cur = make_backend(ctx)(prob, params, aux, opts, True)
    ll_e, st_e, ns_e, cur_e = host(prob, params, aux, opts, True)
    assert np.all(st & _capi.ST_FLOORED) and not np.any(st & 7)
    np.testing.assert_array_equal(st, st_e)
    np.testing.assert_allclose(cur, cur_e, rtol=5e-7)
    np.testing.assert_allclose(ll, ll_e, rtol=1e-6)
    g = orc.Grid(gc.LENGTH, nx, t, 4)
    _, units, idx = gc._names_units("std")
    for m, (c, k) in enumerate(zip(gc.split(prob, cur[0]), firsts)):
        np.testing.assert_allclose(c[:k], free[m][:k], rtol=1e-12)
        assert np.all(c[k:] == min_y[m]) and c[k - 1] > min_y[m]
        g.min_y = min_y[m]
        ref = orc.simulate(gc.seam_profile(nx), g, gc.state_of("std", "stiff"), idx, units=units, RTOL=1e-10,
                           ATOL=1e-16)
        assert np.all(ref[k:] == min_y[m]) and ref[k - 1] > min_y[m]
        assert np.max(np.abs(c[:k] / ref[:k] - 1)) <= gc.SEAM_CURVE_TOL["stiff"]
        want = orc.curve_loglik(c, t, t, prob.vals[prob.t_off[m]:prob.t_off[m] + len(t)],
                                prob.uncs[prob.t_off[m]:prob.t_off[m] + len(t)], gc.SIGMA)
        assert abs(ll[0, m, 0] / want - 1) <= 1e-12, (m, ll[0, m, 0], want)
