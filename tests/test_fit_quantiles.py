"""CPU tier: the per-point quantiles of trpl_fit_quantiles through the host lock-step build of its
selection (csrc/fit_quantiles.h), bit for bit against np.nanquantile(..., method="linear"), and the
draw selection and per-measurement cutting of predictive.posterior_predictive with an injected
evaluator."""
import os
import re
import tempfile
import warnings

import numpy as np
import pytest

from metrotrpl_b200 import _capi
from metrotrpl_b200.predictive import posterior_predictive, select_draws
from metrotrpl_b200.sim_utils import Ensemble
from tests.emu import quantiles_emu as emu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LEVELS = np.array([0.0, 1e-3, 0.025, 0.5, 0.975, 1.0])


def nanquantile(fit, q):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)          # all-NaN columns
        return np.nanquantile(fit, q, axis=0, method="linear")


def check(fit, q):
    quant, count = emu.fit_quantiles(fit, q)
    np.testing.assert_array_equal(quant, nanquantile(fit, q))
    np.testing.assert_array_equal(count, (~np.isnan(fit)).sum(axis=0))
    return quant, count


def as_columns(cols):
    """Columns of different lengths as one [rows, n_cols] buffer, NaN below each column."""
    n = max(1, max(len(c) for c in cols))
    out = np.full((n, len(cols)), np.nan)
    for k, c in enumerate(cols):
        out[:len(c), k] = c
    return out


def adversarial_columns(rng):
    tiny = np.nextafter(1.0, 2.0)
    cols = [[], [3.5], [-2.0, 7.0], [1.0, 1.0], [5.0] * 37, [0.0, -0.0, 0.0, -0.0],
            [np.inf], [-np.inf, np.inf], [np.inf, np.inf], [-np.inf, -np.inf, -np.inf], [1.0, np.inf],
            [-np.inf, 1.0, 2.0], [-np.inf, 0.5, np.inf, 2.0, np.inf], [-1e308, 1e308], [1e308, 1e308, -1e308],
            [1.0, tiny, 1.0, tiny, np.nextafter(1.0, 0.0)], np.nextafter(1.0, 2.0 * np.arange(1, 40)),
            [5e-324, -5e-324, 0.0], np.float64(1.0) + np.arange(17) * np.finfo(float).eps,
            rng.standard_normal(3), rng.standard_normal(100), rng.integers(-3, 4, 200).astype(float),
            rng.choice([-np.inf, np.inf, 0.0, 1.0], 50)]
    return [np.asarray(c, dtype=float) for c in cols]


@pytest.mark.parametrize("levels", ["fixed", "random"])
def test_adversarial_columns_equal_numpy(levels):
    rng = np.random.default_rng(11)
    q = LEVELS if levels == "fixed" else np.sort(rng.random(8))
    check(as_columns(adversarial_columns(rng)), q)
    for lv in q:                    # one level at a time too: each level's own targets
        check(as_columns(adversarial_columns(rng)), [lv])


def test_nan_at_random_places_and_on_a_varying_prefix():
    """IRF curves are compared on a prefix that changes from state to state: NaN past it."""
    rng = np.random.default_rng(5)
    fit = rng.normal(2.0, 0.3, (3000, 61))
    fit[rng.random(fit.shape) < 0.1] = np.nan
    check(fit, LEVELS)
    fit = rng.normal(2.0, 0.3, (3000, 61))
    n_c = rng.integers(0, 62, 3000)
    fit[np.arange(61)[None, :] >= n_c[:, None]] = np.nan
    fit[:, 60] = np.nan                                         # a point no draw compared
    quant, count = check(fit, np.concatenate([LEVELS, rng.random(2)]))
    assert count[60] == 0 and np.all(np.isnan(quant[:, 60]))


def test_large_random_columns():
    rng = np.random.default_rng(9)
    fit = np.concatenate([rng.standard_normal((10000, 8)), rng.lognormal(0, 5, (10000, 8)),
                          np.round(rng.standard_normal((10000, 8)), 1)], axis=1)
    fit[rng.random(fit.shape) < 0.01] = np.nan
    check(fit, LEVELS)
    check(fit, rng.random(8))


def test_refusals():
    fit = np.zeros((4, 3))
    with pytest.raises(ValueError, match="n_q must be in 1..TRPL_MAX_QUANTILES"):
        emu.fit_quantiles(fit, np.linspace(0, 1, _capi.MAX_QUANTILES + 1))
    with pytest.raises(ValueError, match="n_q must be in 1..TRPL_MAX_QUANTILES"):
        emu.fit_quantiles(fit, [])
    for bad in (-1e-300, 1.5, np.nan):
        with pytest.raises(ValueError, match=r"quantile levels must lie in \[0, 1\]"):
            emu.fit_quantiles(fit, [0.5, bad])


def test_header_declares_the_entry_point_and_the_library_exports_it():
    src = open(os.path.join(ROOT, "include", "metrotrpl_b200.h")).read()
    assert re.search(r"int trpl_fit_quantiles\(trpl_handle\* h, int32_t n_q, const double\* q, double\* quant, "
                     r"int32_t\* count\);", src)
    assert int(re.search(r"#define TRPL_MAX_QUANTILES (\d+)", src).group(1)) == _capi.MAX_QUANTILES
    assert hasattr(_capi.load_library(), "trpl_fit_quantiles")


# --- posterior_predictive with an injected evaluator ---

NAMES = ["n0", "p0", "tauN"]


def ensemble(temps=(1.0, 2.0, 1.0), n_iter=40, latest=30, n_t=(7, 5)):
    tmp = tempfile.mkdtemp()
    param_info = {"names": list(NAMES), "active": {n: 1 for n in NAMES}, "unit_conversions": {},
                  "do_log": {n: 1 for n in NAMES}, "prior_dist": {n: (0, np.inf) for n in NAMES},
                  "init_guess": {"n0": 1e8, "p0": 1e15, "tauN": 100.0}, "trial_move": {n: 0.05 for n in NAMES}}
    MCMC = {"init_cond_path": "x", "measurement_path": "y", "output_path": tmp, "num_iters": n_iter,
            "solver": ("solveivp",), "model": "std", "ini_mode": "density", "log_y": 1, "checkpoint_freq": n_iter,
            "model_uncertainty": {"TRPL": 0.1}, "parallel_tempering": list(temps)}
    sim = {"lengths": [300] * len(n_t), "nx": [32] * len(n_t), "meas_types": ["TRPL"] * len(n_t), "num_meas": len(n_t)}
    ms = Ensemble(param_info, sim, MCMC, n_iter)
    ef = ms.ensemble_fields
    rng = np.random.default_rng(1)
    ef["_times"] = [np.linspace(0, 10, n) for n in n_t]
    ef["_vals"] = [rng.normal(2, 0.5, n) for n in n_t]
    ef["_uncs"] = [np.full(n, 0.05) for n in n_t]
    # state k of chain c encodes (c, k), so the evaluator can tell which draws it was given
    ms.H.states[:, 0, :] = np.arange(len(temps))[:, None]
    ms.H.states[:, 1, :] = np.arange(n_iter)[None, :]
    ms.latest_iter = latest
    return ms


def test_draws_come_from_the_cold_chains_after_burn_in():
    ms = ensemble()
    c, k = select_draws(ms, burn_in=0.5, thin=3)
    want_k = np.arange(15, 30, 3)
    np.testing.assert_array_equal(c, np.repeat([0, 2], want_k.size))
    np.testing.assert_array_equal(k, np.tile(want_k, 2))
    c, k = select_draws(ms, burn_in=0.1, thin=1)                # ceil(0.1 * 30) = 3
    assert k.min() == 3 and k.max() == 29 and set(c) == {0, 2}
    c1, k1 = select_draws(ms, burn_in=0.0, max_draws=11, seed=4)
    c2, k2 = select_draws(ms, burn_in=0.0, max_draws=11, seed=4)
    np.testing.assert_array_equal(c1, c2)
    np.testing.assert_array_equal(k1, k2)
    keep = np.sort(np.random.default_rng(4).choice(60, 11, replace=False))
    np.testing.assert_array_equal(c1, np.repeat([0, 2], 30)[keep])
    np.testing.assert_array_equal(k1, np.tile(np.arange(30), 2)[keep])
    c, k = select_draws(ms, burn_in=0.5, max_draws=1000)        # fewer draws than max_draws: all of them
    assert c.size == 30


def test_posterior_predictive_cuts_and_covers_as_numpy_does():
    ms = ensemble()
    ef = ms.ensemble_fields
    q = (0.1, 0.5, 0.9)
    rng = np.random.default_rng(3)
    seen = {}

    def evaluator(states):
        seen["states"] = states.copy()
        n = len(states)
        fit = np.concatenate([v[None, :] + rng.normal(0, 0.6, (n, v.size)) for v in ef["_vals"]], axis=1)
        fit[:, 5:7] = np.nan                                    # measurement 0: last two points never compared
        fit[: n // 2, 10:] = np.nan                             # measurement 1: a shorter prefix for half the draws
        status = np.zeros((n, 2), dtype=np.int32)
        status[0, 1] = _capi.ST_CONV_FAIL
        status[1, 0] = _capi.ST_FLOORED                         # not a failure
        seen["fit"] = fit
        return (*emu.fit_quantiles(fit, q), status)

    res = posterior_predictive(ms, quantiles=q, burn_in=0.5, thin=2, evaluator=evaluator)
    c, k = select_draws(ms, burn_in=0.5, thin=2)
    np.testing.assert_array_equal(seen["states"], ms.H.states[c, :, k])
    np.testing.assert_array_equal(seen["states"][:, 0], c)
    assert res["n_draws"] == len(c) and res["n_failed"] == 1
    np.testing.assert_array_equal(res["quantiles"], q)
    fit = seen["fit"]
    off = 0
    for m, meas in enumerate(res["measurements"]):
        n_t = ef["_times"][m].size
        f = fit[:, off:off + n_t]
        off += n_t
        cmp = (~np.isnan(f)).sum(axis=0) > 0
        np.testing.assert_array_equal(meas["times"], ef["_times"][m][cmp])
        np.testing.assert_array_equal(meas["vals"], ef["_vals"][m][cmp])
        np.testing.assert_array_equal(meas["uncs"], ef["_uncs"][m][cmp])
        np.testing.assert_array_equal(meas["count"], (~np.isnan(f[:, cmp])).sum(axis=0))
        band = nanquantile(f[:, cmp], q)
        np.testing.assert_array_equal(meas["quantiles"], band)
        v = ef["_vals"][m][cmp]
        assert meas["coverage"] == np.mean((v >= band[0]) & (v <= band[-1]))
    assert res["measurements"][0]["times"].size == 5 and res["measurements"][1]["times"].size == 5


def test_posterior_predictive_refuses_bad_arguments():
    ms = ensemble()

    def never(states):
        raise AssertionError("evaluated despite bad arguments")
    for kw, msg in (({"quantiles": ()}, "1 to 8 levels"), ({"quantiles": tuple(np.linspace(0, 1, 9))}, "1 to 8 levels"),
                    ({"quantiles": (0.5, 1.2)}, r"in \[0, 1\]"), ({"quantiles": (np.nan,)}, r"in \[0, 1\]"),
                    ({"quantiles": (0.9, 0.1)}, "ascending"), ({"burn_in": 1.0}, "burn_in"),
                    ({"burn_in": -0.1}, "burn_in"), ({"thin": 0}, "thin"), ({"thin": 1.5}, "thin"),
                    ({"max_draws": 0}, "max_draws")):
        with pytest.raises(ValueError, match=msg):
            posterior_predictive(ms, evaluator=never, **kw)
    with pytest.raises(ValueError, match="no chain at temperature 1"):
        posterior_predictive(ensemble(temps=(1.5, 2.0)), evaluator=never)
    ms.latest_iter = 1
    with pytest.raises(ValueError, match="no draws"):
        posterior_predictive(ms, burn_in=0.5, evaluator=never)
