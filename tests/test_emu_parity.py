"""CPU tier: the kernel's own integrator source, compiled for the host in lock-step (tests/emu),
against the oracle, the golden fixtures and closed forms.  This validates the warp algorithm
(partition + PCR block-tridiagonal solve, RODAS4 controller, Hermite readout, in-kernel
likelihood) without a GPU; the GPU tier (test_gpu_parity.py) repeats every case through the C ABI.
"""
import numpy as np
import pytest

from tests import parity_cases as pc
from tests.emu import emu


def backend(prob, params, aux, opts, want_curves):
    return emu.loglik_batch(prob, params, aux, opts, want_curves)


def test_staub_fixture_rtol_1e7():
    rep = pc.check_staub(backend, rtol=1e-7)
    print(rep)


def test_real_staub_data_three_curves():
    print(pc.check_real3(backend, rtol=1e-7))


def test_known_answers_of_reference_tests():
    print(pc.check_known_answers(backend))


def test_reference_unit_test_parameter_sets():
    print(pc.check_reference_unit_cases(backend))


def test_closed_forms():
    print(pc.check_analytic(backend))


def test_ragged_and_fluence_inputs():
    assert pc.check_edges(backend)


def test_traps_model_with_irf_convolution_nx256():
    print(pc.check_traps_irf(backend))


def test_irf_pass_on_uneven_measurement_times():
    print(pc.check_irf_uneven_times(backend))


def test_team_grids_of_129_to_512_nodes():
    print(pc.check_team_grids(backend))


def test_explicit_rk_path_for_nonstiff_trajectories():
    print(pc.check_explicit_path(backend))


def test_hmax_is_honoured_on_request():
    print(pc.check_hmax_option(backend))


def test_extrapolation_integrator_against_the_converged_truth():
    """csrc/extrapolation.h (order-6 extrapolated linearly implicit Euler), one-warp driver, on both
    staub fixtures; route (A) of the truth is RODAS4 at rtol 1e-9: two unrelated integrators."""
    from metrotrpl_b200 import _capi

    def seulex(prob, params, aux, opts, want_curves):
        o = _capi.SolverOpts(opts.rtol, opts.atol, opts.hmax, opts.max_steps, opts.flags | _capi.OPT_EXTRAPOLATION)
        return emu.loglik_batch(prob, params, aux, o, want_curves)
    for check in (pc.check_staub, pc.check_real3):
        rep = check(seulex, rtol=1e-7, tight_rtol=1e-9, curve_tol=3e-5, truth_backend=backend)
        print({k: v for k, v in rep.items() if not k.startswith("logll_rows")})
        assert rep["mean_steps"] < 200


def _seulex_backend(prob, params, aux, opts, want_curves):
    from metrotrpl_b200 import _capi
    o = _capi.SolverOpts(opts.rtol, opts.atol, opts.hmax, opts.max_steps, opts.flags | _capi.OPT_EXTRAPOLATION)
    return emu.loglik_batch(prob, params, aux, o, want_curves)


def test_extrapolation_integrator_closed_forms_and_ragged_inputs():
    """The one-warp driver of the extrapolation integrator is generic in nodes per lane and model:
    closed forms (nx = 100), ragged curve lengths, fluence mode both ways, nx = 16 / 200 with padding,
    the traps model at nx = 100, the reference's known answers and unit-test parameter sets."""
    print(pc.check_analytic(_seulex_backend))
    assert pc.check_edges(_seulex_backend)
    print(pc.check_known_answers(_seulex_backend))
    print(pc.check_reference_unit_cases(_seulex_backend))


def test_extrapolation_integrator_traps_model_with_irf_convolution_nx256():
    print(pc.check_traps_irf(_seulex_backend, curve_tol=5e-6))     # measured 1.1e-6 (RODAS4: 3e-7)


def test_outputs_without_curves_equal_those_with_curves():
    """The IRF convolution, the min_y floor and the tempering ladder take the likelihood from the
    stored curve, so the run stores it whether or not the caller asked for it, as the library's runs
    do: logll, status, nsteps and ladder rows are bit-identical with and without curves.  traps_irf
    fixture, first two states."""
    from metrotrpl_b200 import _capi
    g = np.load(pc.os.path.join(pc.GOLDEN, "traps_irf.npz"))
    idx = {str(x): i for i, x in enumerate(g["names"])}
    sim = {"lengths": list(g["lengths"]), "nx": [int(g["nx"])] * 2, "meas_types": ["TRPL"] * 2, "num_meas": 2}
    params = _capi.pack_params(g["states"][:2], idx, g["units"], model="traps")
    aux = _capi.default_aux(2, 2, [1.0] * 2, temps=(1.0, 2.0, 4.0))
    ladder = np.array([1.0, 3.0, 9.0])
    for irf, flags in ((True, 0), (False, _capi.OPT_FORCE_MIN_Y), (False, _capi.OPT_LADDER)):
        prob = _capi.pack_problem(sim, g["inis"], [g["t"]] * 2, list(g["vals"]), list(g["uncs"]), model="traps",
                                  ini_mode="fluence", irf_convolution=[520, 520] if irf else None,
                                  irf_tables={520: (g["moments"], g["t_irf"])})
        lad = ladder if flags & _capi.OPT_LADDER else None
        opts = _capi.make_opts(RTOL=1e-7, flags=flags)
        with_curves = emu.loglik_batch(prob, params, aux, opts, True, ladder=lad)
        without = emu.loglik_batch(prob, params, aux, opts, False, ladder=lad)
        assert without[3] is None
        for k in (0, 1, 2) + ((4,) if lad is not None else ()):
            np.testing.assert_array_equal(without[k], with_curves[k], err_msg=f"irf={irf} flags={flags} output {k}")
