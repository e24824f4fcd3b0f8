#!/usr/bin/env python
"""bench.py - TRPL forward simulations per second (nx=128, FP64), BASELINE.json's metric.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--sets S]
                    [--dump-outputs DIR]

Workload (config.workload): BASELINE configs[1] - 4096 random parameter sets (log-uniform in the
prior box of the reference's Inputs/mcmc0.txt, as Dense_Sample/dense_sampling.py:17-35 draws them)
x the 6 TRPL curves of the staub_MAPI_threepower_twothick example (nx=128, 119 measurement times
each), 'std' model, PER GPU (weak scaling: every rank evaluates its own 4096 sets).  One "step" is
one pass of the hot path over that batch: 24576 forward simulations + likelihoods.  The parameter
sets are drawn from fixed seeds and the measurement is stored (tests/golden/bench_measurement.npz),
so the inputs are the same from run to run and from build to build.

value   device-timed throughput, inputs resident in HBM (CUDA events on the library's stream)
e2e     the same through the public API with HOST numpy buffers (H2D + kernel + D2H inside)
The JSON line also carries the FP64 roofline of the trajectory kernel and a CPU baseline (the
oracle port of the reference's numba+SciPy LSODA path, all host cores) timed in the same run.
"""
import argparse
import json
import multiprocessing as mp
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NAMES = "n0 p0 mu_n mu_p ks Cn Cp Sf Sb tauN tauP eps Tm m".split()
UNITS = np.array([1e-21, 1e-21, 1e5, 1e5, 1e12, 1e33, 1e33, 0.01, 0.01, 1, 1, 1, 1, 1.0])
GUESS = np.array([1e8, 3e15, 20, 20, 4.8e-11, 4.4e-29, 4.4e-29, 10, 10, 511, 871, 10, 300, 1.0])
LO = np.array([1e8, 1e14, 1, 1, 1e-11, 1e-29, 1e-29, 1e-4, 1e-4, 1, 1, 10, 300, 1.0])
HI = np.array([1e8, 1e16, 100, 100, 1e-9, 1e-27, 1e-27, 1e4, 1e4, 1500, 3000, 10, 300, 1.0])
IDX = {n: i for i, n in enumerate(NAMES)}
LENGTHS = [311.0, 2000.0, 311.0, 2000.0, 311.0, 2000.0]
NX = 128
SIGMA = 1.0
RTOL = 1e-7   # the reference's default RTOL (forward_solver.py:18)

# Algorithmic FP64 flops of one integrator step per space node, 'std' model, 4 nodes per lane
# (FMA = 2, division = 1); the breakdown is derived in DESIGN.md section 5:
#   6 right-hand sides x 32 + Jacobian 38 (reuses the stage-1 right-hand side's recombination terms
#   and flux factors) + factorisation 184 + 6 solves x 52.5 + stage combinations / error norm 114
#   + readout 8
FLOPS_PER_NODE_STEP = 6 * 32 + 38 + 184 + 6 * 52.5 + 114 + 8   # = 851


def workload_inputs():
    g = np.load(os.path.join(ROOT, "tests", "golden", "staub6.npz"))
    return g["ini"], g["t"]


def draw_states(n_sets, seed):
    rng = np.random.default_rng(seed)
    return 10 ** rng.uniform(np.log10(LO), np.log10(HI), size=(n_sets, len(NAMES)))


def make_shared_fields(ini, t, vals, uncs):
    sim = {"num_meas": 6, "lengths": LENGTHS, "nx": [NX] * 6, "meas_types": ["TRPL"] * 6}
    return {"_sim_info": sim, "_init_params": ini, "_times": [t] * 6, "_vals": vals, "_uncs": uncs,
            "_param_indexes": IDX, "units": UNITS, "model": "std", "ini_mode": "density", "hmax": 4,
            "rtol": RTOL, "atol": None, "solver": ("solveivp",)}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device = device
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.device), f"--query-gpu={self.Q}",
                 "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------
# CPU baseline: the oracle port of the reference path (numba RHS + SciPy LSODA + likelihood)
# ---------------------------------------------------------------------------------------------
_W = {}
REF_DIR = os.path.join(ROOT, "oracle", "_ref")


def ref_available():
    """oracle/_ref holds the unmodified reference modules (oracle/make_ref.py, build container)."""
    return all(os.path.exists(os.path.join(REF_DIR, f)) for f in
               ("trial_move_evaluation.py", "forward_solver.py", "utils.py", "laplace.py", "sim_utils.py"))


def cpu_kind():
    return "reference" if ref_available() else "port"


def _cpu_init(ini, t, vals, uncs):
    # one worker process per core, one thread each: LSODA's dense LU must not spawn BLAS threads
    for k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[k] = "1"
    try:
        from threadpoolctl import threadpool_limits
        _W["tp"] = threadpool_limits(1)
    except Exception:
        pass
    _W.update(ini=ini, t=t, vals=vals, uncs=uncs)
    tt = np.linspace(0, 1, 3)
    sim = {"num_meas": 1, "lengths": [311.0], "nx": [16], "meas_types": ["TRPL"]}
    if ref_available():
        # the reference's own eval_trial_move, unmodified (numba RHS + SciPy LSODA + likelihood)
        import logging
        sys.path.insert(0, REF_DIR)
        import trial_move_evaluation as ref_tme
        _W.update(ref=ref_tme, logger=logging.getLogger("reference"))
        sf = make_shared_fields([1e15 * np.ones(16)], tt, [np.ones(3)], [np.ones(3)])
        sf["_sim_info"] = sim
        sf["_times"], sf["_vals"], sf["_uncs"] = [tt], [np.ones(3)], [np.ones(3)]
        ref_tme.eval_trial_move(GUESS.copy(), {"model_uncertainty": {"TRPL": 1.0}, "_T": 1}, sf, _W["logger"])
    else:
        from oracle import trpl_oracle as orc
        _W.update(orc=orc)
        orc.state_loglik(GUESS, sim, [1e15 * np.ones(16)], [tt], [np.ones(3)], [np.ones(3)], IDX, UNITS,
                         {"TRPL": 1.0})   # numba JIT warm-up, untimed


def _cpu_one(state):
    t = _W["t"]
    if "ref" in _W:
        sf = make_shared_fields(np.array(_W["ini"], dtype=float), t, _W["vals"], _W["uncs"])
        sf["rtol"], sf["atol"] = None, None          # the reference's defaults: 1e-7 / 1e-10, hmax = 4
        ll, _ = _W["ref"].eval_trial_move(np.array(state, dtype=float), {"model_uncertainty": {"TRPL": SIGMA}, "_T": 1},
                                          sf, _W["logger"])
        return ll
    orc = _W["orc"]
    sim = {"num_meas": 6, "lengths": LENGTHS, "nx": [NX] * 6, "meas_types": ["TRPL"] * 6}
    ll, _ = orc.state_loglik(state, sim, _W["ini"], [t] * 6, _W["vals"], _W["uncs"], IDX, UNITS,
                             {"TRPL": SIGMA}, rtol=None, atol=None)
    return ll


def cpu_throughput(states, ini, t, vals, uncs, cores, pool=None):
    """sims/s of the CPU path over `states` (6 curves each) with `cores` worker processes (a work
    queue of single parameter sets: no core waits for another until the queue is empty)."""
    own = pool is None
    if own:
        pool = mp.get_context("fork").Pool(cores, initializer=_cpu_init, initargs=(ini, t, vals, uncs))
        pool.map(_noop, range(cores * 2))
    t0 = time.perf_counter()
    list(pool.imap_unordered(_cpu_one, list(states), chunksize=1))
    dt = time.perf_counter() - t0
    if own:
        pool.close()
    return 6 * len(states) / dt, dt


def _noop(i):
    time.sleep(0.05)
    return i


# ---------------------------------------------------------------------------------------------
def dist_setup(n_gpus):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist_mod
        torch.cuda.set_device(local)
        dist_mod.init_process_group(backend="nccl", device_id=torch.device("cuda", local))
        dist = dist_mod
    return rank, world, local, dist


def allreduce_max(dist, local, x):
    if dist is None:
        return x
    import torch
    tns = torch.tensor([x], dtype=torch.float64, device=f"cuda:{local}")
    dist.all_reduce(tns, op=dist.ReduceOp.MAX)
    return float(tns.item())


def gather_rows(dist, local, row):
    """[world, len(row)] on every rank (diagnostics only)."""
    if dist is None:
        return [list(map(float, row))]
    import torch
    t = torch.tensor(row, dtype=torch.float64, device=f"cuda:{local}")
    out = [torch.empty_like(t) for _ in range(dist.get_world_size())]
    dist.all_gather(out, t)
    return [o.cpu().tolist() for o in out]


def barrier(dist, local):
    if dist is not None:
        import torch
        dist.barrier(device_ids=[local])
        torch.cuda.synchronize(local)


def workload_measurement():
    """Measurement = simulated curves of the initial guess, log10, renoised (like staub's renoised
    file): this project's kernel at rtol 1e-7, plus 0.02 x default_rng(1234).standard_normal per
    curve; uncertainty 0.02.  It is stored rather than simulated at start-up, so that what a build
    is given does not depend on that build's own arithmetic."""
    g = np.load(os.path.join(ROOT, "tests", "golden", "bench_measurement.npz"))
    return list(g["vals"]), list(g["uncs"])


DUMP_LIMIT_BYTES = 60 << 20    # array data; with the .npy headers a dump stays under 64 MB


def dump_outputs(out_dir, arrays):
    """Write each [n_sets, ...] array as out_dir/<name>.npy in float64, plus set_index.npy: the
    parameter sets the rows belong to.  That is every set, or a fixed, seeded sample of them when
    every set would exceed DUMP_LIMIT_BYTES."""
    n_sets = len(next(iter(arrays.values())))
    row_bytes = 8 * (1 + sum(a[0].size for a in arrays.values()))
    keep = np.arange(n_sets)
    if n_sets * row_bytes > DUMP_LIMIT_BYTES:
        keep = np.sort(np.random.default_rng(0).choice(n_sets, DUMP_LIMIT_BYTES // row_bytes, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in dict(arrays, set_index=np.arange(n_sets)).items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.asarray(a, dtype=np.float64)[keep])


def run_ours(args):
    from metrotrpl_b200 import _capi
    from metrotrpl_b200 import trial_move_evaluation as tme
    from metrotrpl_b200.forward_solver import get_context

    rank, world, local, dist = dist_setup(args.gpus)
    ini, t = workload_inputs()
    ctx = get_context(local)
    info = ctx.device_info()
    vals, uncs = workload_measurement()
    sf = make_shared_fields(ini, t, vals, uncs)
    cache = tme.PathCache(sf, device=local)
    states = draw_states(args.sets, seed=20261018 + rank)        # every rank its own shard
    temps = np.ones((args.sets, 3))
    params, aux = cache.pack(states, {"TRPL": SIGMA}, temps)
    sf["rtol"] = args.rtol
    opts = cache.opts()
    n_traj = args.sets * 6

    peak_tf, _ = ctx.fp64_peak_probe(40000)
    launches0 = ctx.launch_count()

    # ---- device-resident throughput -------------------------------------------------------
    ctx.upload(params, aux)
    for _ in range(args.warmup):
        ctx.flush_l2()
        ctx.run_resident(opts)
    ctx.synchronize()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    barrier(dist, local)
    kernel_ms = []
    l_before = ctx.launch_count()
    ctx.timer_begin()
    for _ in range(args.steps):
        ctx.flush_l2()
        ctx.run_resident(opts)
        kernel_ms.append(ctx.last_kernel_ms())
    total_ms = ctx.timer_end()
    gpu_launches = ctx.launch_count() - l_before
    barrier(dist, local)
    clocks = sampler.stop() if rank == 0 else None
    ll, status, nsteps, _ = ctx.download()
    step_ms = allreduce_max(dist, local, total_ms / args.steps)
    value = world * n_traj / (step_ms * 1e-3)
    per_rank = gather_rows(dist, local, [total_ms / args.steps, float(np.mean(kernel_ms)), float(nsteps.sum())])

    # ---- end to end through the public API (host numpy in, host numpy out) ----------------
    for _ in range(max(1, args.warmup // 2)):
        tme.eval_trial_moves(states, temps, {"TRPL": SIGMA}, sf, cache=cache)
    barrier(dist, local)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        res = tme.eval_trial_moves(states, temps, {"TRPL": SIGMA}, sf, cache=cache)
    e2e_s = (time.perf_counter() - t0) / args.steps
    e2e_s = allreduce_max(dist, local, e2e_s)
    e2e_value = world * n_traj / e2e_s
    h2d = params.nbytes + aux.nbytes
    d2h = res.per_meas.nbytes + res.status.nbytes + res.nsteps.nbytes

    # ---- roofline of the trajectory kernel (FP64 pipe; HBM traffic is negligible) ----------
    steps_total = float(nsteps.sum())                               # accepted + rejected
    flops = steps_total * NX * FLOPS_PER_NODE_STEP
    k_ms = float(np.mean(kernel_ms))
    achieved = flops / (k_ms * 1e-3) / 1e12
    alg_bytes = h2d + d2h + ini.nbytes + 3 * 6 * len(t) * 8
    # DRAM traffic per launch cannot be measured without a profiler: it is the committed figure of
    # the last `ncu --set full` capture of this launch size, and says so (traffic_source)
    traffic, traffic_source = None, None
    tpath = os.path.join(ROOT, "profiles", "ncu_dram_traffic.json")
    if os.path.exists(tpath) and args.sets == 4096:
        tj = json.load(open(tpath))
        traffic, traffic_source = tj.get("dram_bytes_per_launch"), "committed ncu figure, not measured in this run: " + tj.get("source", tpath)
    roof = {"bound": "fp64", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s",
            "frac": achieved / peak_tf, "traffic": traffic, "traffic_source": traffic_source,
            "peak_source": "in-run DFMA probe (trpl_fp64_peak_probe); B200 nominal FP64 = 37 TFLOP/s; "
                           "MEASURED_PEAKS.json has no FP64 entry",
            "kernel": "trpl_forward_kernel<4,std>", "kernel_ms": k_ms,
            "flops_per_launch": flops, "flops_per_node_step": FLOPS_PER_NODE_STEP,
            "integrator_steps_per_launch": steps_total,
            "hbm_algorithmic_bytes_per_launch": alg_bytes,
            "hbm_gbs_if_all_traffic_were_dram": alg_bytes / (k_ms * 1e-3) / 1e9}

    # ---- the other BASELINE configs at this N (reported under "extra"; the headline is untouched) --
    extra = None if args.no_extras else run_extras(args, rank, world, local, dist, ini, t, vals, uncs, peak_tf)

    if rank != 0:
        if dist is not None:
            dist.barrier(device_ids=[local])
            dist.destroy_process_group()
        return
    if dist is not None:
        dist.barrier(device_ids=[local])
    # ---- CPU baseline on the host cores (rank 0, N=1 semantics: a bounded sample) ----------
    cores = os.cpu_count() or 1
    n_cpu_sets = max(cores, min(args.cpu_sets, 6 * cores))
    cpu_states = states[:n_cpu_sets]
    if args.no_cpu_baseline or world > 1:      # the CPU baseline is an N=1 figure
        cpu_val, cpu_dt, n_cpu_sets = None, 0.0, 0
    else:
        cpu_val, cpu_dt = cpu_throughput(cpu_states, ini, t, vals, uncs, cores)
    out = {
        "metric": "TRPL forward sims/sec (nx=128, FP64)", "value": value, "unit": "sims/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": workload_config(args, world, len(t)),
        "e2e": {"value": e2e_value, "unit": "sims/s", "h2d_bytes_per_step": int(h2d),
                "d2h_bytes_per_step": int(d2h)},
        "gpu_launches": int(gpu_launches),
        "clocks": clocks,
        "roofline": roof,
        "cpu_baseline": {"value": cpu_val, "unit": "sims/s", "cores": cores, "kind": cpu_kind(),
                         "sample": f"{n_cpu_sets} of the same parameter sets x 6 curves ({cpu_dt:.1f} s wall), "
                                   + CPU_DESCRIPTION[cpu_kind()] + ", rtol 1e-7 / atol 1e-10 / hmax 4 ns"},
        "device": info,
        "extra": extra,
        "stats": {"mean_steps_per_sim": float(nsteps[..., 0].mean()), "max_steps": int(nsteps[..., 0].max()),
                  "mean_rejected": float(nsteps[..., 1].mean()),
                  "frac_floored": float(np.mean((status & 8) != 0)),
                  "frac_failed": float(np.mean((status & 7) != 0)),
                  "kernel_ms_each": [float(x) for x in kernel_ms],
                  "per_rank_[step_ms,kernel_ms,integrator_steps]": per_rank},
    }
    if args.dump_outputs:
        # what a caller of the timed path receives from its last step (Context.download)
        dump_outputs(args.dump_outputs, {"logll": ll, "status": status, "nsteps": nsteps})
    print(json.dumps(out), flush=True)
    if dist is not None:
        dist.destroy_process_group()


def workload_config(args, world, n_t):
    """`config` of the JSON line: the workload the metric is quoted on.  Both arms print the same dict."""
    return {"workload": "configs[1]: 4096 random parameter sets x 6 TRPL curves "
                        "(staub_MAPI threepower_twothick), nx=128, std model, per GPU",
            "sets_per_gpu": args.sets, "curves_per_set": 6, "times_per_curve": int(n_t),
            "rtol": args.rtol, "hmax": "GPU arm: not imposed, steps are error-controlled; reference arm: LSODA "
                                       "with the reference's own max_step = 4 ns (sim_utils.py:17)",
            "l2": "GPU arm: flushed between steps (256 MiB memset); inputs are 0.5 MB and L2-resident by design",
            "parallelism": f"independent parameter-set shards x{world}, no data-path collective"}


CPU_DESCRIPTION = {
    "reference": "the reference's own eval_trial_move (oracle/_ref: unmodified numba RHS + SciPy LSODA + likelihood)",
    "port": "oracle port of the reference's numba RHS + SciPy LSODA + likelihood (oracle/_ref absent)"}


# Algorithmic flops per node and integrator step of the configs[3] instantiation (traps model, two
# warps per trajectory with 4 nodes per lane: csrc/team_kernels.cu), counted like FLOPS_PER_NODE_STEP (DESIGN.md section 5): 6 right-hand sides x 40 +
# Jacobian and trap condensation 54 + factorisation 155 + 6 solves x 53.3 + stage combinations and
# error norm on three components 171 + readout 9.  The IRF convolution is not counted.
FLOPS_PER_NODE_STEP_TRAPS_NX256 = 6 * 40 + 54 + 155 + 6 * 53.3 + 171 + 9   # = 949


def run_extras(args, rank, world, local, dist, ini, t, vals, uncs, peak_tf):
    """configs[2] (parallel tempering, 256 replicas sharded over the ranks), configs[3] (traps + IRF,
    nx = 256, per GPU) and configs[4] (dense grid, sharded) at this N.  Every rank takes part."""
    import tempfile
    from metrotrpl_b200 import _capi
    from metrotrpl_b200 import dense_sampling as ds
    from metrotrpl_b200.metropolis import metro
    from metrotrpl_b200.parallel import Comm
    os.environ["TRPL_USE_LOCAL_RANK"] = "1"
    comm = Comm()
    out = {}
    # ---- configs[3]: traps model + IRF convolution, nx = 256 (weak: every rank its own batch) ----
    g = np.load(os.path.join(ROOT, "tests", "golden", "traps_irf.npz"))
    names = [str(n) for n in g["names"]]
    idx = {n: i for i, n in enumerate(names)}
    tt = g["t"]
    nx = int(g["nx"])
    tables = {520: (g["moments"], g["t_irf"])}
    sim = {"lengths": list(g["lengths"]), "nx": [nx] * 2, "meas_types": ["TRPL"] * 2, "num_meas": 2}
    prob = _capi.pack_problem(sim, g["inis"], [tt] * 2, list(g["vals"]), list(g["uncs"]), model="traps",
                              ini_mode="fluence", irf_convolution=[520, 520], irf_tables=tables)
    n_sets = 4096
    rng = np.random.default_rng(1 + rank)
    base = g["states"][rng.integers(0, len(g["states"]), n_sets)]
    jit = np.ones_like(base)
    act = [idx[n] for n in names if n not in ("n0", "eps", "Tm", "m")]
    jit[:, act] = 10 ** rng.uniform(-0.1, 0.1, size=(n_sets, len(act)))
    params = _capi.pack_params(base * jit, idx, g["units"], model="traps")
    aux = _capi.default_aux(n_sets, 2, [1.0] * 2)
    c3 = _capi.Context(local)
    try:
        c3.set_problem(prob)
        opts = _capi.make_opts(RTOL=1e-7)
        c3.upload(params, aux)
        c3.run_resident(opts)
        c3.synchronize()
        barrier(dist, local)
        ms = []
        c3.timer_begin()
        for _ in range(3):
            c3.flush_l2()
            c3.run_resident(opts)
            ms.append(c3.last_kernel_ms())
        c3.timer_end()
        ll3, st3, ns3, _ = c3.download()
    finally:
        c3.close()
    # device-resident like the headline `value`: the kernel's own events (the L2 flush between the
    # launches is not part of a step), slowest rank
    k_ms = float(np.mean(ms))
    step_ms = allreduce_max(dist, local, k_ms)
    flops = float(ns3.sum()) * nx * FLOPS_PER_NODE_STEP_TRAPS_NX256
    out["traps_nx256_sims_per_s"] = world * 2 * n_sets / (step_ms * 1e-3)
    out["traps_nx256"] = {
        "workload": "configs[3]: traps model + IRF convolution (irf_520nm), nx=256, 4096 parameter sets x 2 curves "
                    "x 401 times per GPU, states jittered +-0.1 decade around the golden fixture's",
        "ms_per_step": step_ms, "mean_steps_per_sim": float(ns3[..., 0].mean()),
        "frac_failed": float(np.mean((st3 & 7) != 0)),
        "roofline": {"bound": "fp64", "achieved": flops / (k_ms * 1e-3) / 1e12, "peak": peak_tf, "unit": "TFLOP/s",
                     "frac": flops / (k_ms * 1e-3) / 1e12 / peak_tf, "kernel": "trpl_team_forward_kernel<4,traps> (two warps per trajectory)",
                     "kernel_ms": k_ms, "flops_per_node_step": FLOPS_PER_NODE_STEP_TRAPS_NX256,
                     "integrator_steps_per_launch": float(ns3.sum()), "traffic": None}}
    # ---- configs[2]: parallel tempering, 256 replicas x 6 curves, swaps every 10 iterations -------
    chains = 256
    param_info = {"names": list(NAMES), "active": {n: int(n not in ("n0", "eps", "Tm", "m")) for n in NAMES},
                  "unit_conversions": dict(zip(NAMES, UNITS)), "do_log": {n: 1 for n in NAMES},
                  "prior_dist": {n: (lo, hi) if lo != hi else (0, np.inf) for n, lo, hi in zip(NAMES, LO, HI)},
                  "init_guess": dict(zip(NAMES, GUESS)), "trial_move": {n: 0.02 for n in NAMES}}
    sim_info = {"num_meas": 6, "lengths": LENGTHS, "nx": [NX] * 6, "meas_types": ["TRPL"] * 6}

    def pt_run(iters, kernel="auto"):
        import copy
        tmp = tempfile.mkdtemp()
        mc = {"init_cond_path": "synthetic", "measurement_path": "synthetic", "output_path": tmp,
              "num_iters": iters, "solver": ("solveivp",), "model": "std", "ini_mode": "density", "log_y": 1,
              "checkpoint_freq": iters, "hard_bounds": 1, "rtol": 1e-7, "atol": None,
              "model_uncertainty": {"TRPL": 0.2}, "parallel_tempering": list(np.logspace(0, 3, chains)),
              "temper_freq": 10}
        comm.barrier()
        t0 = time.perf_counter()
        res = metro(sim_info, ini, ([t] * 6, vals, uncs), mc, copy.deepcopy(param_info), export_path="pt.pik",
                    comm=comm, install_signal_handlers=False, kernel=kernel)
        comm.barrier()
        return time.perf_counter() - t0, res
    short = 11
    pt_run(short)                                                     # warm-up (imports, buffers)
    t_short, _ = pt_run(short)
    t_long, res = pt_run(args.pt_iters)
    rate = (args.pt_iters - short) / max(t_long - t_short, 1e-9)
    rate = 1.0 / allreduce_max(dist, local, 1.0 / rate)
    out["pt_iters_per_s"] = rate
    out["pt"] = {"workload": f"configs[2]: parallel tempering, {chains} replicas x 6 curves (nx=128), swaps every 10 "
                             f"iterations, chains sharded over {world} GPU(s); steady state between iteration "
                             f"{short} and {args.pt_iters}",
                 "sims_per_s": rate * chains * 6, "checksum_logll": float(res.H.loglikelihood[:, -1].sum()),
                 "swap_accept": int(res.H.swap_accept.sum()), "swap_attempts": int(res.H.swap_attempts.sum())}
    # the same chains through the low-latency integrator (order-6 extrapolation, one CTA per
    # trajectory): pays off once an iteration's trajectories fit one wave of a GPU (N >= 4 here)
    pt_run(short, "seulex")
    t_short, _ = pt_run(short, "seulex")
    t_long, res_x = pt_run(args.pt_iters, "seulex")
    rate_x = (args.pt_iters - short) / max(t_long - t_short, 1e-9)
    rate_x = 1.0 / allreduce_max(dist, local, 1.0 / rate_x)
    out["pt_seulex_iters_per_s"] = rate_x
    out["pt"]["seulex_kernel"] = {"iters_per_s": rate_x, "checksum_logll": float(res_x.H.loglikelihood[:, -1].sum()),
                                  "note": "metro(kernel='seulex'): csrc/extrapolation.h; a different integrator, so its "
                                          "chains equal the default kernel's only until a decision differs"}
    # ---- configs[4]: dense grid, args.dense_points per GPU, sharded over the ranks ---------------
    n_pts = args.dense_points * world
    X = draw_states(n_pts, seed=4242)
    sim_flags = {"num_iters": n_pts, "log_y": 1, "model": "std", "ini_mode": "density", "rtol": 1e-7, "atol": None,
                 "likel2move_ratio": {"TRPL": 50.0}, "scale_factor": None, "irf_convolution": None,
                 "current_sigma": {"TRPL": 1.0}, "IRF_tables": None}
    P = np.zeros(n_pts)
    ds.simulate(([t] * 6, vals, uncs), P[:2048 * world].copy(), X[:2048 * world], param_info, dict(sim_info), ini,
                sim_flags, comm=comm)                                 # warm-up
    comm.barrier()
    t0 = time.perf_counter()
    ds.simulate(([t] * 6, vals, uncs), P, X, param_info, dict(sim_info), ini, sim_flags, comm=comm)
    comm.barrier()
    dt = allreduce_max(dist, local, time.perf_counter() - t0)
    out["dense_sims_per_s"] = 6 * n_pts / dt
    out["dense"] = {"workload": f"configs[4]: dense grid, {args.dense_points} points per GPU x 6 curves (nx=128), "
                                f"host buffers in and out, sharded over {world} GPU(s)",
                    "seconds": dt, "n_nonfinite": int((~np.isfinite(P)).sum())}
    return out


def run_reference(args):
    """The reference's CPU path on all host cores: the unmodified reference modules from oracle/_ref
    when present (kind "reference"), else the pinned oracle port.  Each step is a bounded sample of
    the same workload (the first sets of the same seeded parameter-set list the GPU arm draws),
    dealt to the cores from a work queue."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import trpl_oracle as orc
    ini, t = workload_inputs()
    rng = np.random.default_rng(1234)
    sim = {"num_meas": 6, "lengths": LENGTHS, "nx": [NX] * 6, "meas_types": ["TRPL"] * 6}
    cur = [orc.simulate(ini[m], orc.Grid(LENGTHS[m], NX, t, 4), GUESS, IDX, units=UNITS) for m in range(6)]
    vals = [np.log10(cur[m]) + 0.02 * rng.standard_normal(len(t)) for m in range(6)]
    uncs = [np.full(len(t), 0.02) for _ in range(6)]
    cores = os.cpu_count() or 1
    per_step = cores * args.ref_sets_per_core
    states = draw_states(per_step * (args.steps + args.warmup), seed=20261018)
    pool = mp.get_context("fork").Pool(cores, initializer=_cpu_init, initargs=(ini, t, vals, uncs))
    pool.map(_noop, range(cores * 2))
    k = 0
    for _ in range(args.warmup):
        cpu_throughput(states[k:k + per_step], ini, t, vals, uncs, cores, pool=pool)
        k += per_step
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_throughput(states[k:k + per_step], ini, t, vals, uncs, cores, pool=pool)
        k += per_step
    dt = time.perf_counter() - t0
    pool.close()
    value = 6 * per_step * args.steps / dt
    out = {"impl": "reference", "metric": "TRPL forward sims/sec (nx=128, FP64)", "value": value,
           "unit": "sims/s", "n_gpus": int(os.environ.get("WORLD_SIZE", "1")), "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
           # the GPU arm's config, key for key (the workload both arms are quoted on); what this run
           # did with it - a bounded sample per step on the host cores - is under `reference_run`
           "config": workload_config(args, int(os.environ.get("WORLD_SIZE", "1")), len(t)),
           "reference_run": {"sets_per_step": per_step, "rtol": 1e-7, "atol": 1e-10,
                             "hmax": "4 ns (the reference's LSODA max_step, sim_utils.py:17)",
                             "parallelism": f"{cores} worker processes, work queue of single parameter sets"},
           "cpu_baseline": {"value": value, "unit": "sims/s", "cores": cores, "kind": cpu_kind(),
                            "sample": f"{per_step} of the workload's parameter sets x 6 curves per step (the first "
                                      f"ones of the same seeded list), " + CPU_DESCRIPTION[cpu_kind()]},
           "e2e": {"value": value, "unit": "sims/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--sets", type=int, default=4096, help="parameter sets per GPU")
    ap.add_argument("--cpu-sets", type=int, default=48, help="parameter sets in the CPU baseline sample")
    ap.add_argument("--ref-sets-per-core", type=int, default=3)
    ap.add_argument("--no-cpu-baseline", action="store_true", help="profiling runs only")
    ap.add_argument("--rtol", type=float, default=RTOL)
    ap.add_argument("--no-extras", action="store_true", help="skip the configs[2], [3], [4] segments")
    ap.add_argument("--pt-iters", type=int, default=41)
    ap.add_argument("--dense-points", type=int, default=65536, help="dense-grid points per GPU")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed for rank 0's parameter sets "
                         "as DIR/<name>.npy (float64): logll [set, curve, temperature slot], status [set, curve], "
                         "nsteps [set, curve, accepted|rejected], set_index [set]")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU path's outputs (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
