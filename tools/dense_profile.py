import sys, os, time, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import bench
from metrotrpl_b200 import dense_sampling as ds, _capi
from metrotrpl_b200.parallel import Comm
comm = Comm()
ini, t = bench.workload_inputs()
vals, uncs = bench.workload_measurement()
names = bench.NAMES
param_info = {"names": list(names), "active": {n: int(n not in ("n0", "eps", "Tm", "m")) for n in names},
              "unit_conversions": dict(zip(names, bench.UNITS)), "do_log": {n: 1 for n in names},
              "prior_dist": {n: (lo, hi) for n, lo, hi in zip(names, bench.LO, bench.HI)},
              "init_guess": dict(zip(names, bench.GUESS)), "trial_move": {n: 0.02 for n in names}}
sim_info = {"num_meas": 6, "lengths": bench.LENGTHS, "nx": [bench.NX] * 6, "meas_types": ["TRPL"] * 6}
n_pts = 65536
X = bench.draw_states(n_pts, seed=4242)
sim_flags = {"num_iters": n_pts, "log_y": 1, "model": "std", "ini_mode": "density", "rtol": 1e-7, "atol": None,
             "likel2move_ratio": {"TRPL": 50.0}, "scale_factor": None, "irf_convolution": None,
             "current_sigma": {"TRPL": 1.0}, "IRF_tables": None}
# instrument the context calls
orig = {}
acc = {}
def wrap(name):
    f = getattr(_capi.Context, name); orig[name] = f
    def g(self, *a, **k):
        t0 = time.perf_counter(); r = f(self, *a, **k); acc[name] = acc.get(name, 0) + time.perf_counter() - t0; return r
    setattr(_capi.Context, name, g)
for n in ("upload", "run_resident", "download", "set_problem_if_needed", "set_problem", "close", "__init__"):
    wrap(n)
for rep in range(3):
    acc.clear()
    P = np.zeros(n_pts)
    t0 = time.perf_counter()
    ds.simulate(([t] * 6, vals, uncs), P, X, param_info, dict(sim_info), ini, sim_flags, comm=comm)
    dt = time.perf_counter() - t0
    print(json.dumps({"seconds": dt, "sims_per_s": 6 * n_pts / dt, **{k: round(v, 4) for k, v in acc.items()}}))
