"""Posterior predictive bands: what the device quantiles cost against the fit download plus NumPy.

For staub6 (6 curves x 119 points, 'std', nx = 128, RODAS4 one warp per trajectory) and traps_irf
(2 curves x 401 points, traps + IRF, nx = 256, two-warp team) at 10^3, 10^4 and 10^5 jittered
states, one JSON line each:
  fit_launch_ms      the TRPL_OPT_FIT launch (trajectory and fit kernels), CUDA events
  quantile_call_ms   one fit_quantiles call (kernel, copy of the results, stream synchronisation),
                     CUDA events around `reps` calls after a warm-up call
  quantile_kernel_ms fit_quantiles_kernel alone, device time from torch.profiler over `reps` calls
  host_ms            download_fit + np.nanquantile(..., method="linear") on the host, for comparison
Every line also says whether the device result equals the host's bit for bit.  The first line is the
card's name and power limit, read in the same run.

    python tools/predictive_probe.py [--draws 1000 10000 100000] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from metrotrpl_b200 import _capi                                    # noqa: E402
from tests import parity_cases as pc                                # noqa: E402
from tests.test_fit_curves import traps_irf_case                    # noqa: E402

Q = (0.025, 0.5, 0.975)


def fixture(name, n, seed=1):
    rng = np.random.default_rng(seed)
    if name == "staub6":
        g, prob, params, aux = pc.staub_problem()
        names, width = ("tauN", "tauP", "Sf", "Sb", "ks"), 0.1
    else:
        prob, params, aux, _ = traps_irf_case(nx=256, n=4)
        names, width = ("tauN", "tauP", "Nt", "kC"), 0.3
    p = params[np.arange(n) % len(params)].copy()
    for k in names:
        p[:, _capi.PARAM_SLOTS.index(k)] *= 10 ** rng.normal(0, width, n)
    return prob, p, np.repeat(aux[:1], n, axis=0)


def kernel_ms(ctx, reps):
    """Mean device time of fit_quantiles_kernel over reps calls (torch.profiler, CUDA activity)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            ctx.fit_quantiles(Q)
    us = [e.device_time for e in prof.events() if "fit_quantiles_kernel" in e.name]
    return round(sum(us) / len(us) / 1e3, 4) if us else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--draws", type=int, nargs="+", default=[1000, 10000, 100000])
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = []
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    lines.append({"gpu": gpu})
    print(json.dumps(lines[-1]), flush=True)
    ctx = _capi.Context(0)
    for name in ("staub6", "traps_irf"):
        for n in args.draws:
            prob, params, aux = fixture(name, n)
            ctx.set_problem(prob)
            ctx.upload(params, aux)
            ctx.run_resident(_capi.make_opts(RTOL=1e-7, flags=_capi.OPT_FIT))
            ctx.synchronize()
            fit_ms = ctx.last_kernel_ms()
            quant, count = ctx.fit_quantiles(Q)                      # warm-up
            ctx.timer_begin()
            for _ in range(args.reps):
                ctx.fit_quantiles(Q)
            call_ms = ctx.timer_end() / args.reps
            k_ms = kernel_ms(ctx, args.reps)
            t = time.perf_counter()
            fit = ctx.download_fit()
            with warnings.catch_warnings():
                warnings.simplefilter("ignore", RuntimeWarning)
                want = np.nanquantile(fit, Q, axis=0, method="linear")
            host_ms = 1e3 * (time.perf_counter() - t)
            lines.append({
                "fixture": name, "draws": n, "points_per_draw": prob.n_times_total,
                "fit_bytes": int(fit.nbytes), "fit_launch_ms": round(fit_ms, 3),
                "quantile_call_ms": round(call_ms, 4), "quantile_kernel_ms": k_ms, "host_ms": round(host_ms, 1),
                "bit_identical": bool(np.array_equal(quant, want, equal_nan=True)
                                      and np.array_equal(count, (~np.isnan(fit)).sum(axis=0))),
                "points_without_draws": int((count == 0).sum()),
            })
            print(json.dumps(lines[-1]), flush=True)
            del fit, want
    ctx.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("".join(json.dumps(l) + "\n" for l in lines))


if __name__ == "__main__":
    main()
