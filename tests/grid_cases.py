"""Node-count cases shared by the CPU tier (host lock-step build) and the GPU tier (C ABI).  A *backend*
is the callable of parity_cases.py:

    backend(prob, params, aux, opts, want_curves) -> (logll[n_sets,n_meas,3], status, nsteps, curves)

The library runs every curve of a problem on the kernel its largest grid selects (launch_npl in
csrc/trpl_kernels.cu, dispatch in tests/emu/trpl_emu.cpp):

    largest nx   2..32     33..64    65..128    129..256        257..512
    kernel       one warp  one warp  one warp   two-warp team   four-warp team
    nodes/lane   1         2         4          4               4

make_mask (csrc/model.h) gives each lane its nodes: the front contact is node 0 on lane 0, the back
contact node nx-1, and the nodes past it are padding.  Values cross lane seams by shuffles and warp
seams (nodes 127/128, 255/256, 383/384 of a team) through the team mailbox.  The profiles below put a
10x step and two-node peaks on exactly those seams, and on the last real node, so that a term landing
on the wrong node, a value taken from the wrong neighbour or a padding node treated as real changes
the curves far beyond integrator error.

The integrator under test runs at rtol 1e-8 and is held to two truths:
  - the oracle's LSODA on the bit-exact right-hand side (rtol 1e-10, atol 1e-16), over the points
    within two decades of each curve's start.  Below that this LSODA run is itself off: on the
    'fast' row by 1e-7 at three decades and up to 4e-5 at six (measured at nx = 2..128 against LSODA
    at rtol 1e-12 / atol 1e-20, which agrees with the kernel at rtol 1e-11 to 2e-9 over six decades
    at nx = 2 and 33, but takes 36 s per curve at nx = 512).  Seam and contact errors are percent-level
    in the first decade already;
  - the same integrator at rtol 1e-10, over the points within six decades (self-convergence: the
    deep tail of the fast row).
"""
import numpy as np
import pytest

from metrotrpl_b200 import _capi
from oracle import trpl_oracle as orc
from tests import parity_cases as pc

SEAM_NX = (2, 3, 31, 32, 33, 63, 64, 65, 127, 128, 129, 132, 255, 256, 257, 260, 511, 512)
TRAPS_NX = (2, 33, 65, 129, 257, 512)
MIXED = ((127, 100), (200, 128, 65), (400, 100, 129, 257), (512, 40, 5))
LENGTH = 1000.0
T = np.linspace(0, 60, 121)
RTOL = 1e-8
DECADES_LSODA = 2.0
DECADES_SELF = 6.0
TIGHT_RTOL = 1e-10
SIGMA = 1.0
MEAS = ("TRPL", "TRTS")

# Bounds, about 10x the worst value measured on the host lock-step build (measured in brackets).
# vs LSODA, top two decades, any nx, model and readout, per parameter row
SEAM_CURVE_TOL = {"stiff": 3e-8, "fast": 1e-7, "nonstiff": 1e-7}     # [2.9e-9, 8.2e-9, 1.2e-8]
SEAM_SELF_TOL = 4e-7         # rtol 1e-8 vs rtol 1e-10, top six decades                      [4.1e-8]
SEAM_LOGLL_TOL = 5e-9        # relative, vs the oracle's likelihood of the LSODA curve       [5.3e-10]
REVERSAL_TOL = 1e-7          # reversed profile with swapped contacts vs the original  (check_edges) [4.3e-14]
MIXED_NPL_TOL = 1e-13        # another nodes-per-lane count than solo, top three decades     [7.3e-15]
FULL_PADDED_TOL = 1e-12      # padding-free vs padded instantiation on the B200, six decades [4.1e-14]

BASE = dict(pc.BASE, n0=1e8, p0=3e15, ks=4.8e-11, Cn=4.4e-29, Cp=4.4e-29, tauN=511, tauP=871,
            kC=1e-8, Nt=1e15, tauE=50.0)
ROWS = {
    # stiff Rosenbrock path, contacts two decades apart so that swapping them is visible
    "stiff": dict(BASE, mu_n=20, mu_p=20, Sf=10, Sb=1e3),
    # short lifetimes and a fast back contact: more than six decades of decay in the window, the
    # deep tail well below the compared range
    "fast": dict(BASE, mu_n=20, mu_p=20, Sf=10, Sb=1e4, tauN=2, tauP=3),
    # no transport, no contacts: classified non-stiff, explicit Runge-Kutta kernel ('std' only)
    "nonstiff": dict(BASE, mu_n=0, mu_p=0, Sf=0, Sb=0, tauN=4, tauP=6, p0=1e17),
}


def nodes_per_lane(max_nx):
    return 1 if max_nx <= 32 else 2 if max_nx <= 64 else 4


def rows_of(model):
    return ("stiff", "fast", "nonstiff") if model == "std" else ("stiff", "fast")


def _names_units(model):
    names, units, _ = pc._known_units()
    if model == "traps":
        names = names + ["kC", "Nt", "tauE"]
        units = np.concatenate([units, [1e12, 1e-21, 1.0]])
    return names, units, {n: i for i, n in enumerate(names)}


def state_of(model, row, **over):
    names, _, _ = _names_units(model)
    r = dict(ROWS[row], **over)
    return np.array([r[n] for n in names], dtype=float)


def params_of(model, states):
    _, units, idx = _names_units(model)
    return _capi.pack_params(np.atleast_2d(states), idx, units, model=model)


def seams(nx):
    """(step, peaks): the node a 10x step starts at and the first nodes of the seams that carry a
    two-node peak (the node before the seam and the node after it).  The step sits on the last warp
    seam below nx, or for nx <= 128 on the lane seam nearest the middle."""
    npl = nodes_per_lane(nx)
    lane_seam = max(1, (nx // 2) // npl * npl)            # first node of the lane nearest the middle
    warp_seams = [w for w in (128, 256, 384) if w < nx]
    step = warp_seams[-1] if warp_seams else lane_seam
    peaks = sorted({lane_seam} | set(warp_seams) - {step})
    return step, peaks


def seam_profile(nx):
    """Initial excess density [cm^-3]: exp(-x/150), a 10x drop at the step seam, peaks of 4x on the
    two nodes around every other seam and 3x on the last two real nodes."""
    x = (np.arange(nx) + 0.5) * (LENGTH / nx)
    prof = 2e16 * np.exp(-x / 150.0)
    step, peaks = seams(nx)
    prof[step:] *= 0.1
    for s in peaks:
        prof[s - 1:s + 1] *= 4.0
    prof[max(0, nx - 2):] *= 3.0
    return prof


def fake_vals(meas):
    """Measurement values the likelihood compares with: a straight decay in log10, of the order of
    the simulated signals, so that the residuals are O(1)."""
    return (15.0 if meas == "TRPL" else -3.0) - T / 30.0


def pack(nxs, meas, profiles=None, min_y=None, times=None, model="std"):
    tt = T if times is None else times
    sim = {"lengths": [LENGTH] * len(nxs), "nx": list(nxs), "meas_types": list(meas), "num_meas": len(nxs)}
    prof = [seam_profile(n) for n in nxs] if profiles is None else profiles
    vals = [np.interp(tt, T, fake_vals(m)) for m in meas]
    uncs = [np.full(len(tt), 0.05) for _ in meas]
    return _capi.pack_problem(sim, prof, [tt] * len(nxs), vals, uncs, model=model, min_y=min_y)


def split(prob, curves_row):
    return [curves_row[prob.t_off[m]:prob.t_off[m] + prob.n_t[m]] for m in range(prob.n_meas)]


def window_err(mine, ref, decades=DECADES_LSODA):
    """Largest relative error over the points within `decades` of the curve's start."""
    ok = np.abs(ref) >= 10.0 ** (-decades) * np.abs(ref[0])
    return float(np.max(np.abs(mine[ok] / ref[ok] - 1)))


class References:
    """LSODA curves of the seam profiles, computed on first use and kept: one integration gives both
    readouts (PL and photoconductivity come from the same densities)."""

    def __init__(self):
        self._c = {}

    def __call__(self, model, nx, row, meas):
        key = (model, nx, row)
        if key not in self._c:
            _, units, idx = _names_units(model)
            s = state_of(model, row) * units
            g = orc.Grid(LENGTH, nx, T, 4)
            pl, data = orc.simulate(seam_profile(nx), g, state_of(model, row), idx, units=units, model=model,
                                    RTOL=1e-10, ATOL=1e-16, return_fields=True)
            N, P = data[:, :nx], data[:, (1 if model == "std" else 2) * nx:(2 if model == "std" else 3) * nx]
            tr = orc.trts_signal(g.dx, N, P, s[idx["mu_n"]], s[idx["mu_p"]], s[idx["n0"]], s[idx["p0"]]) * 1e9
            low = np.argmax(tr < g.min_y)                       # the floor orc.simulate applies
            if tr[low] < g.min_y:
                tr[low:] = g.min_y
            self._c[key] = {"TRPL": pl, "TRTS": tr}
        return self._c[key][meas]


def _host_agrees(host, prob, params, opts, got):
    """Two compilers, one source: curves to 5e-7, log-likelihoods to 1e-6, steps within 5
    (test_gpu_matches_host_lockstep_build), over the six decades the integrator controls: below them
    the 'fast' row is rounding noise on either side, and so is the likelihood of such a curve."""
    aux = _capi.default_aux(params.shape[0], prob.n_meas, [SIGMA] * prob.n_meas)
    ll_e, st_e, ns_e, cur_e = host(prob, params, aux, opts, True)
    for s in range(params.shape[0]):
        for m, (c, e) in enumerate(zip(split(prob, got[3][s]), split(prob, cur_e[s]))):
            assert window_err(c, e, DECADES_SELF) <= 5e-7, (prob.meas[m].nx, s, m)
            if np.all(e >= 10.0 ** (-DECADES_SELF) * e[0]):
                np.testing.assert_allclose(got[0][s, m], ll_e[s, m], rtol=1e-6)
    assert np.abs(got[2][..., 0] - ns_e[..., 0]).max() <= 5
    keep = 7 | _capi.ST_EXPLICIT
    np.testing.assert_array_equal(got[1] & keep, st_e & keep)


def check_node_count_seams(backend, refs, host=None):
    """Every node count the dispatch distinguishes (first and last grid of each kernel, the lane,
    warp and padding seams on either side), TRPL and TRTS from one profile, three parameter rows
    ('std') and two ('traps'), against LSODA.  Also the in-kernel log-likelihood of the stiff TRPL
    curve against the oracle's likelihood of the LSODA curve.  Measured on the host lock-step build
    (worst over every nx): see the bounds at the top of this module."""
    worst = {}
    cases = [("std", nx) for nx in SEAM_NX] + [("traps", nx) for nx in TRAPS_NX]
    for model, nx in cases:
        rows = rows_of(model)
        prob = pack([nx, nx], MEAS, model=model)
        params = params_of(model, [state_of(model, r) for r in rows])
        aux = _capi.default_aux(len(rows), 2, [SIGMA] * 2)
        opts = _capi.make_opts(RTOL=RTOL)
        got = backend(prob, params, aux, opts, True)
        ll, st, ns, cur = got
        cur_t = backend(prob, params, aux, _capi.make_opts(RTOL=TIGHT_RTOL), True)[3]
        assert not np.any(st & 7), (model, nx, st)
        for r, row in enumerate(rows):
            explicit = bool(np.all(st[r] & _capi.ST_EXPLICIT))
            assert explicit == (row == "nonstiff") and (explicit or not np.any(st[r] & _capi.ST_EXPLICIT)), \
                (model, nx, row, st[r])
            for c, c_t, meas in zip(split(prob, cur[r]), split(prob, cur_t[r]), MEAS):
                e = window_err(c, refs(model, nx, row, meas))
                e_t = window_err(c, c_t, DECADES_SELF)
                for key, v in ((f"{model}/{meas}/nx{nx}", e), (f"{model}/{meas}/nx{nx}/self", e_t)):
                    worst[key] = max(worst.get(key, 0.0), v)
                assert e <= SEAM_CURVE_TOL[row] and e_t <= SEAM_SELF_TOL, (model, nx, row, meas, e, e_t)
        want = orc.curve_loglik(refs(model, nx, "stiff", "TRPL"), T, T, fake_vals("TRPL"), np.full(len(T), 0.05),
                                SIGMA)
        rel = abs(ll[0, 0, 0] / want - 1)
        worst[f"{model}/logll/nx{nx}"] = rel
        assert rel <= SEAM_LOGLL_TOL, (model, nx, ll[0, 0, 0], want)
        if host is not None:
            _host_agrees(host, prob, params, opts, got)
    return worst


def check_reversal_with_swapped_contacts(backend):
    """A film lit from the back with the contacts swapped is the same film: the reversed seam profile
    with Sf and Sb exchanged gives the curves of the original, TRPL and TRTS.  At nx = 33 and 511 the
    back contact sits on a lane with padding behind it, at 129 and 257 the first node of a warp holds
    the back contact; reversing moves the sharp features to the other side of every seam."""
    out = {}
    for nx in (33, 129, 257, 511):
        p = seam_profile(nx)
        prob = pack([nx, nx, nx, nx], ["TRPL", "TRPL", "TRTS", "TRTS"], profiles=[p, p[::-1], p, p[::-1]])
        fwd, rev = state_of("std", "stiff"), state_of("std", "stiff", Sf=ROWS["stiff"]["Sb"], Sb=ROWS["stiff"]["Sf"])
        _, st, ns, cur = backend(prob, params_of("std", [fwd, rev]), _capi.default_aux(2, 4, [SIGMA] * 4),
                                 _capi.make_opts(RTOL=RTOL, flags=_capi.OPT_NO_LIKELIHOOD), True)
        assert not np.any(st & 7), (nx, st)
        a, b = split(prob, cur[0]), split(prob, cur[1])
        worst = 0.0
        for m, mr in ((0, 1), (1, 0), (2, 3), (3, 2)):
            worst = max(worst, float(np.max(np.abs(b[mr] / a[m] - 1))))
        # the same physics with the contacts where they were is a different curve: the check has teeth
        assert np.max(np.abs(a[1] / a[0] - 1)) > 100 * REVERSAL_TOL
        assert worst <= REVERSAL_TOL, (nx, worst)
        out[nx] = worst
    return out


def check_mixed_grids(backend, refs, host=None, fma_contracted=False):
    """Grids of several sizes in one problem: every curve runs on the kernel of the largest grid, the
    smaller ones with padding lanes (and, in a team, padding warps) behind their back contact.  Each
    curve equals the same measurement run alone, with the same step counts: bit for bit where both
    kernels hold four nodes per lane (the elimination order is the same), within MIXED_NPL_TOL where
    the solo run holds one or two (40 and 5 nodes; measured 7e-15).  Each also matches LSODA.

    fma_contracted: the backend is compiled with a*b+c contracted into FMAs (nvcc).  A grid of 128 or
    512 nodes alone runs on the padding-free instantiation, where every mask but the contact lanes is
    a compile-time constant and the selects vanish (make_mask), so the compiler sees other expressions
    and contracts them differently: rounding-level differences, FULL_PADDED_TOL, same step counts.
    Measured on the B200: nx = 128 (one warp alone, two-warp team in [200, 128, 65]) bit-identical;
    nx = 512 in [512, 40, 5] bit-identical on the stiff row, 3.6e-15 on the fast row's curve and
    4.1e-14 on its likelihood.  The host build (-ffp-contract=off) is bit-identical in both."""
    out, differ = {}, []
    rows = ("stiff", "fast")
    params = params_of("std", [state_of("std", r) for r in rows])
    opts = _capi.make_opts(RTOL=RTOL)
    for nxs in MIXED:
        meas = [MEAS[i % 2] for i in range(len(nxs))]
        prob = pack(nxs, meas)
        aux = _capi.default_aux(len(rows), len(nxs), [SIGMA] * len(nxs))
        got = backend(prob, params, aux, opts, True)
        ll, st, ns, cur = got
        assert not np.any(st & 7), (nxs, st)
        npl = nodes_per_lane(max(nxs))
        for m, nx in enumerate(nxs):
            solo_prob = pack([nx], [meas[m]])
            s_ll, s_st, s_ns, s_cur = backend(solo_prob, params, _capi.default_aux(len(rows), 1, [SIGMA]), opts, True)
            np.testing.assert_array_equal(ns[:, m], s_ns[:, 0], err_msg=f"{nxs} nx={nx}")
            np.testing.assert_array_equal(st[:, m], s_st[:, 0], err_msg=f"{nxs} nx={nx}")
            for r, row in enumerate(rows):
                c, s = split(prob, cur[r])[m], s_cur[r]
                d_ll = float(np.max(np.abs(ll[r, m] / s_ll[r, 0] - 1)))
                if nodes_per_lane(nx) == npl and fma_contracted and nx in (128, 512):
                    d = window_err(c, s, DECADES_SELF)
                    out[f"{nxs}/nx{nx}/{row}"] = (d, d_ll)
                    assert d <= FULL_PADDED_TOL and d_ll <= FULL_PADDED_TOL, (nxs, nx, row, d, d_ll)
                elif nodes_per_lane(nx) == npl:
                    # the likelihood sums are reduced over the lanes of the kernel (64 or 128 in a
                    # team): another lane count, another summation order
                    if not np.array_equal(c, s) or d_ll > 1e-14:
                        differ.append((nxs, nx, row, window_err(c, s, DECADES_SELF), d_ll))
                else:
                    d = window_err(c, s, 3.0)
                    out[f"{nxs}/nx{nx}/{row}"] = d
                    assert d <= MIXED_NPL_TOL, (nxs, nx, row, d)
                e = window_err(c, refs("std", nx, row, meas[m]))
                assert e <= SEAM_CURVE_TOL[row], (nxs, nx, row, e)
        if host is not None:
            _host_agrees(host, prob, params, opts, got)
    assert not differ, differ          # every case first, so that one run shows the whole pattern
    return out


def check_grid_refusals(backend):
    """The two contacts must sit on different lanes (model.h computes one contact term per lane), so a
    problem whose smallest grid has no more nodes than a lane of its largest grid's kernel holds is
    refused, as is a grid outside 2..512 nodes.  The smallest grids just above the limit run."""
    params = params_of("std", [state_of("std", "stiff")])
    opts = _capi.make_opts(RTOL=RTOL, flags=_capi.OPT_NO_LIKELIHOOD)
    for nxs, msg in (((512, 4), "mixed nx"), ((200, 3), "mixed nx"), ((64, 2), "mixed nx"),
                     ((1,), r"nx must be in 2\.\.512"), ((513,), r"nx must be in 2\.\.512"),
                     ((128, 1), r"nx must be in 2\.\.512")):
        prob = pack(nxs, ["TRPL"] * len(nxs), profiles=[np.full(n, 1e16) for n in nxs])
        with pytest.raises(RuntimeError, match=msg):
            backend(prob, params, _capi.default_aux(1, len(nxs), [SIGMA] * len(nxs)), opts, True)
    for nxs in ((512, 5), (64, 3)):
        prob = pack(nxs, ["TRPL"] * len(nxs))
        _, st, _, cur = backend(prob, params, _capi.default_aux(1, len(nxs), [SIGMA] * len(nxs)), opts, True)
        assert not np.any(st & 7), (nxs, st)
        assert np.all(np.isfinite(cur)) and np.all(cur > 0), nxs
    return True
