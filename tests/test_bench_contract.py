"""CPU tier: the reference arm of bench.py (the reference's CPU path on the host cores) runs
without a GPU and prints the contract's JSON line; the inputs are fixed and --dump-outputs writes
what the timed path computed (GPU tier for the run itself)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    env = dict(os.environ, RANK="0", WORLD_SIZE="1")
    out = subprocess.check_output([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference",
                                   "--steps", "1", "--warmup", "0", "--ref-sets-per-core", "1"], text=True,
                                  env=env, timeout=600)
    line = json.loads(out.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "sims/s" and line["higher_is_better"] is True
    assert line["metric"] == "TRPL forward sims/sec (nx=128, FP64)"
    assert line["value"] > 0 and line["steps"] == 1
    # oracle/_ref (the unmodified reference modules, oracle/make_ref.py) when present, else the port
    have_ref = os.path.exists(os.path.join(ROOT, "oracle", "_ref", "trial_move_evaluation.py"))
    assert line["cpu_baseline"]["kind"] == ("reference" if have_ref else "port")
    assert line["cpu_baseline"]["cores"] >= 1 and "hmax" in line["config"]
    assert line["e2e"] == {"value": line["value"], "unit": "sims/s", "h2d_bytes_per_step": 0,
                           "d2h_bytes_per_step": 0}
    assert line["config"]["workload"].startswith("configs[1]")


def test_other_ranks_of_the_reference_arm_do_nothing():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.check_output([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference",
                                   "--steps", "1", "--warmup", "0"], text=True, env=env, timeout=120)
    assert out.strip() == ""


def test_stored_measurement_is_the_renoised_initial_guess(golden_dir):
    """bench's measurement is the initial guess's curves (the reference's LSODA at tight tolerance
    agrees with this project's kernel there to ~1e-7 in log10) plus 0.02 x default_rng(1234)."""
    vals, uncs = bench.workload_measurement()
    g = np.load(os.path.join(golden_dir, "staub6.npz"))
    np.testing.assert_array_equal(g["states"][0], bench.GUESS)
    rng = np.random.default_rng(1234)
    for m in range(6):
        noise = 0.02 * rng.standard_normal(len(g["t"]))
        np.testing.assert_allclose(vals[m] - noise, np.log10(g["pl_tight"][0, m]), rtol=0, atol=1e-6)
        np.testing.assert_array_equal(uncs[m], np.full(len(g["t"]), 0.02))


def test_dump_outputs_all_sets_or_a_seeded_sample(tmp_path, monkeypatch):
    ll = np.arange(40 * 6 * 3, dtype=float).reshape(40, 6, 3) - 0.5
    status = np.arange(40 * 6, dtype=np.int32).reshape(40, 6)

    def load(d):
        return {n: np.load(tmp_path / d / f"{n}.npy") for n in ("logll", "status", "set_index")}
    bench.dump_outputs(str(tmp_path / "all"), {"logll": ll, "status": status})
    got = load("all")
    assert all(a.dtype == np.float64 for a in got.values())
    np.testing.assert_array_equal(got["logll"], ll)
    np.testing.assert_array_equal(got["status"], status)
    np.testing.assert_array_equal(got["set_index"], np.arange(40))
    # room for 10 of the 40 sets: the same sorted sample every time, rows and indices together
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 10 * 8 * (18 + 6 + 1))
    bench.dump_outputs(str(tmp_path / "a"), {"logll": ll, "status": status})
    bench.dump_outputs(str(tmp_path / "b"), {"logll": ll, "status": status})
    a, b = load("a"), load("b")
    keep = a["set_index"].astype(int)
    assert len(keep) == 10 and np.all(np.diff(keep) > 0)
    for n in a:
        np.testing.assert_array_equal(a[n], b[n])
    np.testing.assert_array_equal(a["logll"], ll[keep])
    np.testing.assert_array_equal(a["status"], status[keep])


@pytest.mark.gpu
def test_dump_outputs_hold_what_the_timed_steps_computed(tmp_path):
    """--steps sets the number of timed steps, and --dump-outputs writes the last one's results: the
    same numbers the public API gives for the same parameter sets and measurement."""
    from metrotrpl_b200.trial_move_evaluation import eval_trial_moves
    n_sets = 64
    out = subprocess.check_output([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2",
                                   "--warmup", "1", "--sets", str(n_sets), "--no-extras", "--no-cpu-baseline",
                                   "--dump-outputs", str(tmp_path)], text=True, timeout=600)
    line = json.loads(out.strip().splitlines()[-1])
    assert line["steps"] == 2 and len(line["stats"]["kernel_ms_each"]) == 2
    got = {n: np.load(tmp_path / f"{n}.npy") for n in ("logll", "status", "nsteps", "set_index")}
    assert all(a.dtype == np.float64 for a in got.values())
    assert got["logll"].shape == (n_sets, 6, 3) and got["nsteps"].shape == (n_sets, 6, 2)
    np.testing.assert_array_equal(got["set_index"], np.arange(n_sets))
    ini, t = bench.workload_inputs()
    vals, uncs = bench.workload_measurement()
    sf = bench.make_shared_fields(ini, t, vals, uncs)
    res = eval_trial_moves(bench.draw_states(n_sets, seed=20261018), np.ones(n_sets), {"TRPL": bench.SIGMA}, sf)
    np.testing.assert_allclose(got["logll"], res.per_meas, rtol=1e-12, atol=0)
    np.testing.assert_array_equal(got["status"], res.status)
    np.testing.assert_array_equal(got["nsteps"], res.nsteps)
