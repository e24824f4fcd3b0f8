"""Metropolis sampler driver: the reference's metro() with whole batches per iteration.

Reference: metropolis.py.  What changes is *when* likelihoods are computed, not what is computed:

  * reference (serial fallback, metropolis.py:93-137): for each chain in turn - propose, simulate
    num_meas curves on the CPU, accept/reject; tempering swaps re-simulate both partners.
  * here: the proposals of ALL chains of an iteration are drawn first (consuming the generator in
    exactly the reference's serial order: chain m's proposal draws, then chain m's acceptance
    draw), evaluated in ONE kernel launch (n_chains x num_meas trajectories), then accepted or
    rejected.  The kernel also returns every proposal's likelihood at every ladder temperature
    (the reference's ll_funcs), so swaps (metropolis.py:66-90) are pure host arithmetic.
  * several GPUs: chains are sharded over ranks for the launch and the per-chain likelihood rows
    are all-gathered (parallel.Comm); every rank then makes the same accept/swap decisions from
    the same generator state, so results do not depend on the number of GPUs.

One deliberate difference: the reference's serial swap `a[i], a[i+1] = a[i+1], a[i]` on NumPy
views leaves both chains holding the upper chain's state (an aliasing slip; its MPI path swaps
correctly).  Here the states are swapped.
"""
from __future__ import annotations

import os
import pickle
import signal
from time import perf_counter

import numpy as np

from . import _capi
from .laplace import load_irf_tables
from .mcmc_logging import start_logging, stop_logging
from .parallel import Comm
from .sim_utils import Ensemble
from .trial_move_generation import make_trial_move, make_trial_moves

MSG_FREQ = 100       # metropolis.py:31
MSG_COOLDOWN = 3     # metropolis.py:32
SEED = 235817049752375780   # metropolis.py:296


def roll_acceptance(rng, logratio):
    """metropolis.py:35-39."""
    if isinstance(logratio, np.ndarray):
        return rng.random(len(logratio)) < np.exp(logratio)
    return rng.random() < np.exp(logratio)


class CudaEvaluator:
    """Likelihood of a batch of states at every ladder temperature, on this rank's GPU."""

    def __init__(self, shared_fields, device=None, kernel="auto"):
        from .trial_move_evaluation import PathCache
        if kernel not in ("auto", "warp", "cta", "seulex"):
            raise ValueError(f"unknown kernel {kernel!r}")
        # "auto" is RODAS4 with one trajectory per warp.  A tempering iteration is as slow as its
        # slowest trajectory, but measured on B200, RODAS4 on a whole CTA ("cta",
        # csrc/cta_trajectory.h) has the SAME latency per integrator step (6.5 us: a step is a chain
        # of ~50 dependent exchange-and-reduce levels either way, tools/latency_probe.py, DESIGN.md
        # section 5) at 0.3x the throughput.  "seulex" (csrc/extrapolation.h) is a different
        # integrator: log-likelihoods agree with RODAS4's to 2e-7, not bit for bit, so it is never
        # chosen automatically.
        self.kernel = "warp" if kernel == "auto" else kernel
        self.cache = PathCache(shared_fields, device=device, kernel=self.kernel)
        self.ladder = np.ascontiguousarray(shared_fields["_T"], dtype=np.float64)
        self.flags = self.cache.flags | _capi.OPT_LADDER
        self._cost = None       # integrator steps of the previous call's trajectories
        # trajectories this GPU holds at once (148 SMs x 2 CTAs x 4 warps, or x 1 per CTA): a batch
        # that fits starts all at once and the queue order (and the step counts it needs) is moot
        sm = self.cache.ctx.device_info()["sm_count"] if hasattr(self.cache.ctx, "device_info") else 148
        self._resident = sm * 2 * (1 if self.flags & _capi.OPT_CTA_PER_TRAJ else 4)

    def launch(self, states, sigmas):
        """Upload and launch; nothing is waited for.  Returns the number of parameter sets."""
        n = states.shape[0]
        params, aux = self.cache.pack(states, sigmas, np.ones((n, 3)))   # slot 1 = sigma^2 (T = 1)
        sf = self.cache.sf
        opts = _capi.make_opts(sf.get("rtol", None), sf.get("atol", None), flags=self.flags)
        ctx = self.cache.ctx
        ctx.set_problem_if_needed(self.cache.prob)
        # the ladder lives on the (process-wide) context: another evaluator may have replaced it
        if getattr(ctx, "_ladder_key", None) != self.ladder.tobytes():
            ctx.set_ladder(self.ladder)
            ctx._ladder_key = self.ladder.tobytes()
        # Longest first: a chain's proposal costs about what its previous proposal cost, and an
        # iteration is only as fast as its last trajectory.  The order never changes a result.
        self._ordered = n * self.cache.n_meas > self._resident
        if self._ordered and self._cost is not None and self._cost.size == n * self.cache.n_meas:
            ctx.set_queue_order(np.argsort(-self._cost, kind="stable"))
        elif self._ordered or self._cost is not None:
            ctx.set_queue_order(None)
            self._cost = None
        ctx.upload(params, aux)
        ctx.run_resident(opts)
        return n

    def __call__(self, states, sigmas):
        """states [n, n_params], sigmas: list of {meas_type: sigma}.  Returns [n, n_T] on the host
        (one stream synchronisation)."""
        n = self.launch(states, sigmas)
        rows, nsteps = self.cache.ctx.download_ladder_sums(n, want_nsteps=self._ordered)
        if self._ordered:
            self._cost = nsteps.sum(axis=-1).ravel()
        return rows

    def device_rows(self, states, sigmas):
        """Same rows left in HBM: (device pointer, n, n_T).  The step counts (next call's queue
        order) are fetched too."""
        n = self.launch(states, sigmas)
        ptr, n_sets, n_t = self.cache.ctx.ladder_sums_resident()
        if self._ordered:
            self._cost = self.cache.ctx.download_nsteps(n).sum(axis=-1).ravel()
        return ptr, n_sets, n_t


def sharded_eval(evaluator, comm, states, sigmas):
    """Evaluate all chains' states, each rank its own block; every rank gets all rows."""
    n = states.shape[0]
    lo, hi = comm.shard(n)
    if comm.world == 1:
        return evaluator(states, sigmas)
    if comm.backend == "nccl" and hasattr(evaluator, "device_rows"):
        # rows stay in HBM and cross NVLink device to device; one D2H of the gathered table
        ptr, n_local, n_t = evaluator.device_rows(states[lo:hi], sigmas[lo:hi])
        return comm.allgather_device_rows(ptr, n_local, n_t, n)
    local = evaluator(states[lo:hi], sigmas[lo:hi])
    return comm.allgather_rows(local, n)


def main_metro_loop_batched(states, logll, accept, starting_iter, num_iters, shared_fields,
                            unique_fields, RNG, logger, evaluator, comm, cur_ladder=None,
                            need_initial_state=True, reference_swap_aliasing=False):
    """Batched twin of main_metro_loop_serial (metropolis.py:93-137).

    states [n_chains, n_params, n_iters], logll/accept [n_chains, n_iters]; cur_ladder
    [n_chains, n_T] holds each chain's current state's likelihood at every ladder temperature.
    """
    n_chains = shared_fields["_n_chains"]
    T = np.asarray(shared_fields["_T"], dtype=float)
    own = np.arange(n_chains)
    sigmas = [uf["model_uncertainty"] for uf in unique_fields]
    swap_accept = np.zeros(n_chains, dtype=int)
    swap_attempts = np.zeros(n_chains, dtype=int)
    if need_initial_state:
        logger.info("Simulating initial state:")
        cur_ladder = sharded_eval(evaluator, comm, np.ascontiguousarray(states[:, :, 0]), sigmas)
        logll[:, 0] = cur_ladder[own, own]
        starting_iter += 1
    elif cur_ladder is None:
        cur_ladder = sharded_eval(evaluator, comm,
                                  np.ascontiguousarray(states[:, :, starting_iter - 1]), sigmas)
    prof = {"proposals": 0.0, "evaluate": 0.0, "accept": 0.0, "swaps": 0.0} if os.environ.get("TRPL_PT_PROFILE") else None
    for k in range(starting_iter, num_iters):
        t_a = perf_counter()
        if k % MSG_FREQ == 0 or k < starting_iter + MSG_COOLDOWN:
            for m in range(n_chains):
                logger.info(f"Iter {k} MetroState #{m} Current state: {states[m, :, k-1]} logll {logll[m, k-1]}")
        # proposals and acceptance draws in the reference's generator order
        moves = np.sqrt(T)[:, None] * shared_fields["base_trial_move"][None, :]
        # The reference warns for every failed proposal attempt; with hundreds of hot chains that is
        # thousands of lines per iteration.  A one-line summary is written on the iterations whose
        # states are logged anyway (every MSG_FREQ-th and the first few).
        verbose_iter = k % MSG_FREQ == 0 or k < starting_iter + MSG_COOLDOWN
        proposals, u = make_trial_moves(states[:, :, k - 1], moves, shared_fields, RNG, logger if verbose_iter else None)
        t_b = perf_counter()
        new_ladder = sharded_eval(evaluator, comm, proposals, sigmas)
        t_c = perf_counter()
        new_ll = new_ladder[own, own]
        n_bad = int(np.count_nonzero(np.isneginf(new_ll)))
        if n_bad:
            # the reference warns once per failed simulation (trial_move_evaluation.py:66-72, 103-106,
            # 117-123, 159-165); here one line per iteration
            logger.warning(f"Iter {k}: {n_bad} of {n_chains} proposals have likelihood -inf "
                           "(integrator failure, failed convolution, too many negative values or NaN)")
        logratio = new_ll - logll[:, k - 1]
        logratio = np.where(np.isnan(logratio), -np.inf, logratio)
        with np.errstate(over="ignore"):
            accepted = u < np.exp(logratio)
        logll[:, k] = np.where(accepted, new_ll, logll[:, k - 1])
        states[:, :, k] = np.where(accepted[:, None], proposals, states[:, :, k - 1])
        accept[accepted, k] = 1
        cur_ladder[accepted] = new_ladder[accepted]
        t_d = perf_counter()
        if shared_fields["do_parallel_tempering"] and k % shared_fields["temper_freq"] == 0:
            for _ in range(n_chains - 1):
                i = RNG.integers(0, n_chains - 1)
                swap_attempts[i] += 1
                bi_ui, bj_ui = cur_ladder[i, i], cur_ladder[i, i + 1]
                bi_uj, bj_uj = cur_ladder[i + 1, i], cur_ladder[i + 1, i + 1]
                ratio = bi_ui + bj_uj - bi_uj - bj_ui
                with np.errstate(over="ignore", invalid="ignore"):
                    ok = RNG.random() < np.exp(-ratio)
                if ok:
                    swap_accept[i] += 1
                    logll[i, k] = bi_uj
                    logll[i + 1, k] = bj_ui
                    if reference_swap_aliasing:
                        # metropolis.py:86 of the reference: a tuple swap of two NumPy views leaves
                        # BOTH chains with the upper chain's state (and the upper chain's logll entry
                        # with the lower state's likelihood).  Reproduced only on request, to compare
                        # whole chains with the reference's serial path bit for bit.
                        states[i, :, k] = states[i + 1, :, k]
                        cur_ladder[i] = cur_ladder[i + 1]
                    else:
                        tmp = states[i, :, k].copy()
                        states[i, :, k] = states[i + 1, :, k]
                        states[i + 1, :, k] = tmp
                        cur_ladder[[i, i + 1]] = cur_ladder[[i + 1, i]]
        if prof is not None:
            t_e = perf_counter()
            prof["proposals"] += t_b - t_a; prof["evaluate"] += t_c - t_b
            prof["accept"] += t_d - t_c; prof["swaps"] += t_e - t_d
    if prof is not None and num_iters > starting_iter:
        n_it = num_iters - starting_iter
        logger.info("host profile, ms per iteration: " + ", ".join(f"{k_} {1e3 * v / n_it:.3f}" for k_, v in prof.items()))
        print("[trpl] host profile, ms per iteration (rank %d): " % comm.rank + ", ".join(f"{k_} {1e3 * v / n_it:.3f}" for k_, v in prof.items()), flush=True)
    return states, logll, accept, swap_attempts, swap_accept, cur_ladder


def kill_from_cl(signal_n, frame):
    raise KeyboardInterrupt("Terminate from command line")


def all_signal_handler(func):
    for s in signal.Signals:
        try:
            signal.signal(s, func)
        except (ValueError, OSError, RuntimeError):
            continue


def metro(sim_info, iniPar, e_data, MCMC_fields, param_info, verbose=False, export_path="",
          **kwargs):
    """Same call as the reference's metro() (metropolis.py:283-473).

    Extra keyword arguments: evaluator_factory (tests), comm (a parallel.Comm), irf_dir,
    install_signal_handlers (default True, as the reference), kernel ("auto" | "warp" | "cta" | "seulex":
    which instantiation of the integrator evaluates the proposals, see CudaEvaluator),
    reference_swap_aliasing (default False: swap correctly; True reproduces the reference's serial
    swap, metropolis.py:86, which leaves both chains with the upper chain's state).
    """
    clock0 = perf_counter()
    comm = kwargs.get("comm", None) or Comm()
    rank = comm.rank
    if kwargs.get("install_signal_handlers", True):
        all_signal_handler(kill_from_cl)
    os.makedirs(MCMC_fields["output_path"], exist_ok=True)
    load_checkpoint = MCMC_fields.get("load_checkpoint", None)
    num_iters = MCMC_fields["num_iters"]
    checkpoint_freq = MCMC_fields.get("checkpoint_freq", num_iters)
    RNG = np.random.default_rng(SEED)
    logger_name = kwargs.get("logger_name", "Ensemble0") + f"-rank{rank}-"
    logger, handler = start_logging(log_dir=MCMC_fields["output_path"], name=logger_name, verbose=verbose)

    starting_iter = 0
    if load_checkpoint is None:
        MS_list = Ensemble(param_info, sim_info, MCMC_fields, num_iters, verbose)
        ef = MS_list.ensemble_fields
        ef["_init_params"] = iniPar
        ef["_times"], ef["_vals"], ef["_uncs"] = e_data
        MS_list.random_state = RNG.bit_generator.state
        if ef.get("irf_convolution", None) is not None:
            ef["_IRF_tables"] = load_irf_tables(ef["irf_convolution"], kwargs.get("irf_dir", "IRFs"))
        else:
            ef["_IRF_tables"] = {}
        if rank == 0:
            MS_list.checkpoint(os.path.join(ef["output_path"], export_path))
    else:
        with open(os.path.join(MCMC_fields["output_path"], load_checkpoint), "rb") as f:
            MS_list = pickle.load(f)
        if "starting_iter" in MCMC_fields and MCMC_fields["starting_iter"] < MS_list.latest_iter:
            starting_iter = MCMC_fields["starting_iter"]
            MS_list.H.extend(starting_iter)
        else:
            starting_iter = MS_list.latest_iter
            MS_list.H.extend(num_iters)
            MS_list.ensemble_fields["num_iters"] = MCMC_fields["num_iters"]
    shared_fields = MS_list.ensemble_fields
    unique_fields = MS_list.unique_fields
    RNG.bit_generator.state = MS_list.random_state
    states, logll, accept = MS_list.H.states, MS_list.H.loglikelihood, MS_list.H.accept

    if comm.world > shared_fields["_n_chains"]:
        # every rank must own at least one chain; checked here, before any collective, on all ranks
        raise ValueError(f"more ranks ({comm.world}) than chains ({shared_fields['_n_chains']})")
    factory = kwargs.get("evaluator_factory", None)
    evaluator = factory(shared_fields) if factory is not None else CudaEvaluator(
        shared_fields, device=comm.local_rank, kernel=kwargs.get("kernel", "auto"))

    need_initial_state = load_checkpoint is None
    cur_ladder = None
    ending_iter = min(starting_iter + checkpoint_freq, num_iters)
    swap_att = swap_acc = None
    while ending_iter <= num_iters:
        logger.info(f"Simulating from {starting_iter} to {ending_iter}")
        states, logll, accept, swap_att, swap_acc, cur_ladder = main_metro_loop_batched(
            states, logll, accept, starting_iter, ending_iter, shared_fields, unique_fields, RNG, logger,
            evaluator, comm, cur_ladder=cur_ladder, need_initial_state=need_initial_state,
            reference_swap_aliasing=kwargs.get("reference_swap_aliasing", False))
        MS_list.H.swap_attempts += swap_att
        MS_list.H.swap_accept += swap_acc
        if ending_iter == num_iters:
            break
        MS_list.latest_iter = ending_iter
        MS_list.H.pack(states, logll, accept)
        MS_list.random_state = RNG.bit_generator.state
        if rank == 0:
            logger.info(f"Saving checkpoint at k={ending_iter}")
            MS_list.checkpoint(os.path.join(shared_fields["output_path"], export_path))
        need_initial_state = False
        starting_iter = ending_iter
        ending_iter = min(ending_iter + checkpoint_freq, num_iters)
    logger.info(f"Rank {rank} took {perf_counter() - clock0} s")
    MS_list.latest_iter = ending_iter
    MS_list.H.pack(states, logll, accept)
    MS_list.random_state = RNG.bit_generator.state
    if rank == 0:
        logger.info(f"Swap accept rate: {MS_list.H.swap_accept} accepted of {MS_list.H.swap_attempts} attempts")
        logger.info(f"Exporting to {shared_fields['output_path']}")
        MS_list.checkpoint(os.path.join(shared_fields["output_path"], export_path))
    stop_logging(logger, handler, 0)
    return MS_list
