"""Parallel-tempering example at BASELINE configs[2] size: 256 temperature replicas x 6 TRPL curves
(nx = 128), swaps every 10 steps, chains sharded over the ranks of one node.

    python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 tools/run_pt_example.py --iters 30

Prints one JSON line (rank 0): iterations/s, simulations/s, swap statistics.
"""
import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
from metrotrpl_b200.metropolis import metro  # noqa: E402
from metrotrpl_b200.parallel import Comm  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=31)
    ap.add_argument("--chains", type=int, default=256)
    ap.add_argument("--kernel", default="auto", choices=["auto", "warp", "cta", "seulex"])
    args = ap.parse_args()
    comm = Comm()
    ini, t = bench.workload_inputs()
    os.environ["TRPL_USE_LOCAL_RANK"] = "1"
    vals, uncs = bench.workload_measurement()
    names = bench.NAMES
    param_info = {"names": list(names), "active": {n: int(n not in ("n0", "eps", "Tm", "m")) for n in names},
                  "unit_conversions": dict(zip(names, bench.UNITS)), "do_log": {n: 1 for n in names},
                  "prior_dist": {n: (lo, hi) if lo != hi else (0, np.inf) for n, lo, hi in zip(names, bench.LO, bench.HI)},
                  "init_guess": dict(zip(names, bench.GUESS)), "trial_move": {n: 0.02 for n in names}}
    sim_info = {"num_meas": 6, "lengths": bench.LENGTHS, "nx": [bench.NX] * 6, "meas_types": ["TRPL"] * 6}
    out = tempfile.mkdtemp()
    MCMC = {"init_cond_path": "synthetic", "measurement_path": "synthetic", "output_path": out,
            "num_iters": args.iters, "solver": ("solveivp",), "model": "std", "ini_mode": "density",
            "log_y": 1, "checkpoint_freq": args.iters, "hard_bounds": 1, "rtol": 1e-7, "atol": None,
            "model_uncertainty": {"TRPL": 0.2},
            "parallel_tempering": list(np.logspace(0, 3, args.chains)), "temper_freq": 10}
    comm.barrier()
    t0 = time.perf_counter()
    ms = metro(sim_info, ini, ([t] * 6, vals, uncs), MCMC, param_info, export_path="pt.pik", comm=comm,
               install_signal_handlers=False, kernel=args.kernel)
    comm.barrier()
    dt = time.perf_counter() - t0
    if comm.rank == 0:
        sims = args.chains * 6 * args.iters
        print(json.dumps({"workload": "configs[2] parallel tempering", "chains": args.chains, "iters": args.iters,
                          "n_gpus": comm.world, "seconds": dt, "iters_per_s": args.iters / dt,
                          "sims_per_s": sims / dt, "accept_rate": float(ms.H.accept[:, 1:].mean()),
                          "swap_accept": int(ms.H.swap_accept.sum()), "swap_attempts": int(ms.H.swap_attempts.sum()),
                          "checksum_logll": float(ms.H.loglikelihood[:, -1].sum()),
                          "checksum_states": float(np.log10(ms.H.states[:, :, -1]).sum()), "kernel": args.kernel}))


if __name__ == "__main__":
    main()
