"""Adaptive tempered SMC on the six-curve staub problem (tests/golden/staub6.npz, 'std', nx = 128),
against parallel-tempering metro() given the same wall time.

For every active set (2: tauN and Sf, the many-start MLE fixture; 8: p0, mu_n, mu_p, ks, Sf, Sb, tauN,
tauP, each on a box of two decades around the state the data were made with) and every N, smc() runs
through CUDA (RODAS4, one warp per trajectory) and the script prints one JSON line: wall time, stages,
launches, trajectories, the trajectory rate inside the likelihood launches next to the headline rate
of profiles/r02_bench_n1.json, log Z, and effective posterior draws per second (N after the final
resample).  Then metro() with a 256-rung ladder runs for the same wall time on the same problem and
prior box (hard_bounds), and its line gives the autocorrelation ESS of the _T = 1 chain (the second
half of it, smallest over the active parameters) per second.  The first line is the card's name and
power limit, read in the same run.

    python tools/smc_probe.py [--particles 1024 4096 16384] [--active 2 8] [--out FILE]
    python -m torch.distributed.run --nproc-per-node G tools/smc_probe.py --particles 65536 --active 2 --no-metro --out FILE
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

from metrotrpl_b200.metropolis import metro                        # noqa: E402
from metrotrpl_b200.parallel import Comm                           # noqa: E402
from metrotrpl_b200.smc import make_cuda_loglik, smc               # noqa: E402
from tests.test_gpu_mle_multistart import staub_mle_inputs         # noqa: E402

ACTIVE = {2: ("tauN", "Sf"), 8: ("p0", "mu_n", "mu_p", "ks", "Sf", "Sb", "tauN", "tauP")}
LADDER = 256


def inputs(n_active, tmp):
    """smc() / metro() positional arguments: (sim_info, ini, e_data, MCMC, param_info)."""
    e_data, sim_info, param_info, ini, MCMC = staub_mle_inputs(tmp)
    if n_active == 8:
        g = np.load(os.path.join(ROOT, "tests", "golden", "staub6.npz"))
        truth = dict(zip([str(n) for n in g["names"]], g["states"][0]))
        names = ACTIVE[8]
        param_info["active"] = {n: int(n in names) for n in param_info["names"]}
        param_info["prior_dist"].update({n: (truth[n] / 10, truth[n] * 10) for n in names})
        param_info["init_guess"].update({n: truth[n] * 1.5 for n in names})
    return sim_info, ini, e_data, MCMC, param_info


def timed_factory(stats, sigma, kernel, device):
    def factory(ef):
        f = make_cuda_loglik(ef, sigma, device=device, kernel=kernel)

        def loglik(states):
            t = time.perf_counter()
            ll = f(states)                                  # synchronous: the result is on the host
            stats["seconds"] += time.perf_counter() - t
            return ll
        return loglik
    return factory


def autocorr_ess(x):
    """Effective sample size of a chain by Geyer's initial positive sequence of autocorrelations."""
    x = np.asarray(x, dtype=float) - np.mean(x)
    n = len(x)
    if n < 4 or not np.any(x):
        return float("nan")
    f = np.fft.rfft(x, 2 * n)
    acf = np.fft.irfft(f * np.conj(f))[:n]
    acf /= acf[0]
    tau = -1.0
    for k in range(0, n - 1, 2):
        pair = acf[k] + acf[k + 1]
        if pair <= 0:
            break
        tau += 2 * pair
    return n / max(tau, 1.0)


def run_smc(n_active, n, moves, kernel, comm, seed):
    stats = {"seconds": 0.0}
    sim_info, ini, e_data, MCMC, param_info = inputs(n_active, tempfile.mkdtemp())
    comm.barrier()
    t = time.perf_counter()
    ms = smc(sim_info, ini, e_data, MCMC, param_info, n_particles=n, n_moves=moves, seed=seed, comm=comm,
             kernel=kernel, evaluator_factory=timed_factory(stats, MCMC["current_sigma"], kernel, comm.local_rank))
    comm.barrier()
    return ms, time.perf_counter() - t, stats["seconds"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--particles", type=int, nargs="+", default=[1024, 4096, 16384])
    ap.add_argument("--active", type=int, nargs="+", default=[2, 8], choices=sorted(ACTIVE))
    ap.add_argument("--moves", type=int, default=5)
    ap.add_argument("--kernel", default="warp", choices=["warp", "cta", "seulex"])
    ap.add_argument("--no-metro", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    comm = Comm()
    lines = []

    def emit(d):
        if comm.rank == 0:
            lines.append(d)
            print(json.dumps(d), flush=True)
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()
    with open(os.path.join(ROOT, "profiles", "r02_bench_n1.json")) as f:
        headline = json.loads(f.read().strip().splitlines()[-1]).get("value")
    emit({"gpu": gpu[comm.local_rank], "n_gpus": comm.world})
    run_smc(2, 256, 1, args.kernel, comm, 0)                         # warm-up: module load, buffers
    for n_active in args.active:
        for n in args.particles:
            ms, wall, launch_s = run_smc(n_active, n, args.moves, args.kernel, comm, 1)
            st = ms.smc
            traj = int(st["trajectories"].sum())
            emit({"sampler": "smc", "active": list(ACTIVE[n_active]), "n_particles": n, "n_moves": args.moves,
                  "n_gpus": comm.world, "wall_s": round(wall, 3), "stages": len(st["beta"]),
                  "launches": int(st["launches"].sum()), "trajectories": traj,
                  "launch_s_rank0": round(launch_s, 3),
                  "trajectories_per_s_in_launches": round(traj / launch_s, 1),
                  "headline_sims_per_s_1gpu": headline, "log_evidence": st["log_evidence"],
                  "acceptance_final": round(float(st["acceptance"][-1]), 3),
                  "effective_draws": n, "effective_draws_per_s": round(n / wall, 2)})
            if args.no_metro:
                continue
            sim_info, ini, e_data, MCMC, param_info = inputs(n_active, tempfile.mkdtemp())
            mcmc = {k: v for k, v in MCMC.items() if k != "current_sigma"}

            def metro_run(iters):
                m = dict(mcmc, num_iters=iters, checkpoint_freq=iters, hard_bounds=1,
                         model_uncertainty=MCMC["current_sigma"],
                         parallel_tempering=list(np.logspace(0, 3, LADDER)), temper_freq=10)
                pi = {k: (dict(v) if isinstance(v, dict) else v) for k, v in param_info.items()}
                pi["trial_move"] = {k: 0.01 for k in pi["names"]}
                t = time.perf_counter()
                out = metro(sim_info, ini, e_data, m, pi, export_path="pt.pik", comm=comm,
                            install_signal_handlers=False, kernel=args.kernel)
                return out, time.perf_counter() - t
            _, t21 = metro_run(21)                               # the set-up, and the time per iteration
            _, t81 = metro_run(81)
            per_iter = (t81 - t21) / 60
            iters = max(21, int((wall - (t21 - 21 * per_iter)) / per_iter))
            pt, pt_wall = metro_run(iters)
            chain = np.log10(pt.H.states[0][np.asarray(pt.ensemble_fields["active"])][:, iters // 2:])
            ess = min(autocorr_ess(c) for c in chain)
            emit({"sampler": "metro", "active": list(ACTIVE[n_active]), "ladder": LADDER, "trial_move": 0.01,
                  "n_gpus": comm.world, "iterations": iters, "wall_s": round(pt_wall, 3),
                  "smc_wall_s": round(wall, 3), "accept_T1": round(float(pt.H.accept[0, 1:].mean()), 3),
                  "autocorr_ess_T1_second_half": round(ess, 1), "effective_draws_per_s": round(ess / pt_wall, 2)})
    if args.out and comm.rank == 0:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as f:
            f.write("".join(json.dumps(line) + "\n" for line in lines))


if __name__ == "__main__":
    main()
