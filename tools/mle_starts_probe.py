"""Many-start maximum likelihood on the six-curve staub problem: what K starts cost per iteration.

For each K, mle(starts=K, seed=1) through CUDA (RODAS4, one warp per trajectory) runs to the end
and the script prints one JSON line: wall time of the search per iteration of its slowest start,
launches, trajectories per launch, iterations, and the log-likelihood time inside it.  The first
line is the card's name and power limit, read in the same run.

    python tools/mle_starts_probe.py [--starts 1 16 64 256 1024] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from metrotrpl_b200.max_likelihood import mle                       # noqa: E402
from metrotrpl_b200.sim_utils import Ensemble                       # noqa: E402
from metrotrpl_b200.trial_move_evaluation import PathCache, eval_trial_moves   # noqa: E402
from tests.test_gpu_mle_multistart import staub_mle_inputs          # noqa: E402


def counting_evaluator():
    """The CUDA log-likelihood mle() builds by default, with launches, sets and time counted."""
    e_data, sim_info, param_info, ini, MCMC = staub_mle_inputs(tempfile.mkdtemp())
    sigma = MCMC["current_sigma"]
    ef = Ensemble(param_info, sim_info, dict(MCMC, num_iters=1, checkpoint_freq=1), 1).ensemble_fields
    ef["_init_params"] = ini
    ef["_times"], ef["_vals"], ef["_uncs"] = e_data
    ef["_IRF_tables"] = None
    cache = PathCache(ef)
    stats = {"launches": 0, "sets": 0, "seconds": 0.0}

    def evaluator(states):
        t = time.perf_counter()
        ll = eval_trial_moves(states, np.ones(len(states)), sigma, ef, cache=cache).logll   # synchronous
        stats["seconds"] += time.perf_counter() - t
        stats["launches"] += 1
        stats["sets"] += len(states)
        return ll
    return evaluator, stats, cache.n_meas


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--starts", type=int, nargs="+", default=[1, 16, 64, 256, 1024])
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = []
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    lines.append({"gpu": gpu})
    print(json.dumps(lines[-1]), flush=True)
    evaluator, stats, n_meas = counting_evaluator()
    mle(*staub_mle_inputs(tempfile.mkdtemp()), None, None, evaluator=evaluator, starts=4, seed=0)   # warm-up
    for K in args.starts:
        for k in stats:
            stats[k] = 0 if k != "seconds" else 0.0
        t = time.perf_counter()
        ms = mle(*staub_mle_inputs(tempfile.mkdtemp()), None, None, evaluator=evaluator, starts=K, seed=1)
        wall = time.perf_counter() - t
        st = ms.opt.get("starts", {"nit": np.array([ms.opt["nit"]]), "fun": np.array([ms.opt["fun"]])})
        iters = int(st["nit"].max())
        lines.append({
            "starts": K, "iterations": iters, "nit_median": float(np.median(st["nit"])),
            "wall_s": round(wall, 4), "wall_ms_per_iteration": round(1e3 * wall / iters, 3),
            "loglik_ms_per_iteration": round(1e3 * stats["seconds"] / iters, 3),
            "launches": stats["launches"], "trajectories_per_launch": round(stats["sets"] * n_meas / stats["launches"], 1),
            "best_cost": float(ms.opt["fun"]), "start0_cost": float(st["fun"][0]),
            "best_start": int(ms.opt.get("best_start", 0)),
            "distinct_optima": int(len(np.unique(np.round(st["fun"], 6)))),
        })
        print(json.dumps(lines[-1]), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("".join(json.dumps(l) + "\n" for l in lines))


if __name__ == "__main__":
    main()
