"""Dense-sampling example at BASELINE configs[4] size: random parameter points x 6 TRPL curves
(nx = 128), the grid sharded over the ranks of one node (no collective until the final gather).

    python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 tools/run_dense_example.py --points 1000000

Prints one JSON line (rank 0): simulations/s over the whole job, best sample, checksum of the
likelihood vector (identical for every N: each point's result does not depend on the sharding).
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
from metrotrpl_b200 import dense_sampling as ds  # noqa: E402
from metrotrpl_b200.parallel import Comm  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--points", type=int, default=1_000_000)
    ap.add_argument("--block", type=int, default=ds.DEFAULT_BLOCK)
    args = ap.parse_args()
    comm = Comm()
    ini, t = bench.workload_inputs()
    os.environ["TRPL_USE_LOCAL_RANK"] = "1"
    vals, uncs = bench.workload_measurement()
    names = bench.NAMES
    param_info = {"names": list(names), "active": {n: int(n not in ("n0", "eps", "Tm", "m")) for n in names},
                  "unit_conversions": dict(zip(names, bench.UNITS)), "do_log": {n: 1 for n in names},
                  "prior_dist": {n: (lo, hi) for n, lo, hi in zip(names, bench.LO, bench.HI)},
                  "init_guess": dict(zip(names, bench.GUESS)), "trial_move": {n: 0.02 for n in names}}
    sim_info = {"num_meas": 6, "lengths": bench.LENGTHS, "nx": [bench.NX] * 6, "meas_types": ["TRPL"] * 6}
    sim_flags = {"num_iters": args.points, "log_y": 1, "model": "std", "ini_mode": "density", "rtol": 1e-7,
                 "atol": None, "likel2move_ratio": {"TRPL": 50.0}, "scale_factor": None, "irf_convolution": None}
    np.random.seed(20261018)          # every rank draws the same grid (the reference's np.random.uniform)
    names_l = list(names)
    min_X = np.array([bench.LO[names_l.index(n)] for n in names_l])
    max_X = np.array([bench.HI[names_l.index(n)] for n in names_l])
    N, P, X = ds.make_grid(None, None, min_X, max_X, np.ones(len(names_l), dtype=bool), sim_flags)
    sim_flags["current_sigma"] = {"TRPL": 1.0}
    sim_flags["IRF_tables"] = None
    comm.barrier()
    t0 = time.perf_counter()
    ds.simulate(([t] * 6, vals, uncs), P, X, param_info, dict(sim_info), ini, sim_flags, comm=comm, block=args.block)
    comm.barrier()
    dt = time.perf_counter() - t0
    if comm.rank == 0:
        fin = np.isfinite(P)
        print(json.dumps({"workload": "configs[4] dense sampling", "points": args.points, "curves_per_point": 6,
                          "n_gpus": comm.world, "block": args.block, "seconds": dt,
                          "sims_per_s": 6 * args.points / dt, "best_logll": float(P[fin].max()),
                          "argbest": int(np.argmax(np.where(fin, P, -np.inf))),
                          "checksum_logll_finite_sum": float(np.sum(np.maximum(P[fin], -1e12))),
                          "n_nonfinite": int((~fin).sum())}))
    comm.finalize() if hasattr(comm, "finalize") else None


if __name__ == "__main__":
    main()
