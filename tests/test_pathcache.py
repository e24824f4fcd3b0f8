"""CPU tier: host packing of the per-measurement factors (`_s#` scale factors, `_f#` fluence and
`_a#` absorption multipliers, with and without constraint groups) - the lookups of
trial_move_evaluation.py:38-60 of the reference - without a device (the context is a stub)."""
import numpy as np
import pytest

from metrotrpl_b200 import _capi
from metrotrpl_b200.trial_move_evaluation import PathCache


class StubContext:
    def set_problem(self, prob):
        self.problem = prob


def shared_fields(**extra):
    names = ["n0", "p0", "mu_n", "mu_p", "ks", "Cn", "Cp", "Sf", "Sb", "tauN", "tauP", "eps", "Tm", "m",
             "_s0", "_s1", "_f0", "_f1", "_f2", "_f3", "_a0"]
    t = np.linspace(0, 10, 11)
    sim = {"lengths": [300.0] * 4, "nx": [32] * 4, "meas_types": ["TRPL"] * 4, "num_meas": 4}
    sf = {"_sim_info": sim, "_init_params": [np.array([1e12, 6e4, 1.0])] * 4, "_times": [t] * 4,
          "_vals": [np.zeros(11)] * 4, "_uncs": [np.ones(11)] * 4,
          "_param_indexes": {n: i for i, n in enumerate(names)}, "units": np.ones(len(names)),
          "model": "std", "ini_mode": "fluence"}
    sf.update(extra)
    return sf, names


def test_group_lookup_of_scale_fluence_and_absorption_factors():
    sf, names = shared_fields(scale_factor=(0.02, [0, 1, 2, 3], [(0, 2), (1, 3)]),
                              fittable_fluences=(0.02, [0, 1, 3], None),
                              fittable_absps=(0.02, [2], [(0, 2)]))
    cache = PathCache(sf, ctx=StubContext())
    idx = sf["_param_indexes"]
    assert cache.s_idx.tolist() == [idx["_s0"], idx["_s1"], idx["_s0"], idx["_s1"]]      # groups -> first member
    assert cache.f_idx.tolist() == [idx["_f0"], idx["_f1"], -1, idx["_f3"]]              # no groups -> own index
    assert cache.a_idx.tolist() == [-1, -1, idx["_a0"], -1]
    rng = np.random.default_rng(0)
    states = 10 ** rng.uniform(-1, 1, size=(3, len(names)))
    params, aux = cache.pack(states, {"TRPL": 2.0}, np.array([[1.0, 2.0, 4.0]] * 3))
    for m in range(4):
        np.testing.assert_array_equal(aux[:, m, _capi.A_SCALE_SHIFT], np.log10(states[:, cache.s_idx[m]]))
        want_f = states[:, cache.f_idx[m]] if cache.f_idx[m] >= 0 else np.ones(3)
        want_a = states[:, cache.a_idx[m]] if cache.a_idx[m] >= 0 else np.ones(3)
        np.testing.assert_array_equal(aux[:, m, _capi.A_FLUENCE_MULT], want_f)
        np.testing.assert_array_equal(aux[:, m, _capi.A_ABSORB_MULT], want_a)
        np.testing.assert_array_equal(aux[:, m, _capi.A_S2T0:_capi.A_S2T0 + 3], np.array([[4.0, 8.0, 16.0]] * 3))
    # measurements outside the spec's list keep the neutral values
    sf2, _ = shared_fields(scale_factor=(0.02, [1], None))
    c2 = PathCache(sf2, ctx=StubContext())
    assert c2.s_idx.tolist() == [-1, sf2["_param_indexes"]["_s1"], -1, -1]
    _, aux2 = c2.pack(states, {"TRPL": 1.0}, np.ones((3, 3)))
    assert np.all(aux2[:, [0, 2, 3], _capi.A_SCALE_SHIFT] == 0.0)


def test_fittable_initial_condition_factors_are_refused_in_density_mode():
    sf, _ = shared_fields(fittable_fluences=(0.02, [0], None))
    sf["ini_mode"] = "density"
    sf["_init_params"] = [np.ones(32)] * 4
    with pytest.raises(ValueError, match="fluence"):
        PathCache(sf, ctx=StubContext())


def test_pa_measurements_are_refused():
    sf, _ = shared_fields()
    sf["_sim_info"] = dict(sf["_sim_info"], meas_types=["TRPL", "pa", "TRPL", "TRPL"])
    with pytest.raises(NotImplementedError):
        PathCache(sf, ctx=StubContext())


def test_kernel_names_map_to_flags(monkeypatch):
    """PathCache maps "warp" | "cta" | "seulex" to launch flags; CudaEvaluator reads them back and
    runs "auto" as "warp"."""
    from metrotrpl_b200 import metropolis, trial_move_evaluation
    sf, _ = shared_fields(_T=np.array([1.0, 2.0]))
    assert PathCache(sf, ctx=StubContext()).flags == 0
    assert PathCache(sf, ctx=StubContext(), kernel="cta").flags == _capi.OPT_CTA_PER_TRAJ
    with pytest.raises(ValueError, match="unknown kernel"):
        PathCache(sf, ctx=StubContext(), kernel="auto")
    monkeypatch.setattr(trial_move_evaluation, "get_context", lambda device=None: StubContext())
    for name, kernel, flags, resident in (("auto", "warp", 0, 148 * 8), ("warp", "warp", 0, 148 * 8),
                                          ("cta", "cta", _capi.OPT_CTA_PER_TRAJ, 148 * 2)):
        ev = metropolis.CudaEvaluator(sf, kernel=name)
        assert (ev.kernel, ev.flags, ev._resident) == (kernel, flags | _capi.OPT_LADDER, resident)
    with pytest.raises(ValueError, match="unknown kernel"):
        metropolis.CudaEvaluator(sf, kernel="bogus")
