"""Latency of small batches: RODAS4 one warp / one CTA per trajectory, and the order-6 extrapolation
integrator one warp / one CTA per trajectory.
usage (GPU box): python tools/latency_probe.py [--model std|traps] [n_sets ...]

--model std (default): the six staub curves (nx = 128), all four kernels.
--model traps: the traps + IRF problem of tests/golden/traps_irf.npz on 128 nodes, states jittered
+-0.1 decade around the fixture's (as bench.py builds configs[3]); RODAS4 one warp against the
extrapolation integrator one CTA per trajectory (the two kernels that hold the traps model here).
The first line names the card and its power limit."""
import json
import subprocess
import sys

import numpy as np

sys.path.insert(0, ".")
from metrotrpl_b200 import _capi          # noqa: E402
import bench                              # noqa: E402
from tests import parity_cases as pc      # noqa: E402

args = sys.argv[1:]
model = "std"
if "--model" in args:
    k = args.index("--model")
    model = args[k + 1]
    del args[k:k + 2]
if model not in ("std", "traps"):
    raise SystemExit(f"unknown model {model!r}")

ctx = _capi.Context(0)
try:
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True, timeout=60).stdout.strip()
except (OSError, subprocess.SubprocessError):
    smi = "unavailable"
print(json.dumps({"device": ctx.device_info()["name"], "nvidia_smi_name_power_limit": smi, "model": model}),
      flush=True)

if model == "std":
    g, prob, _, _ = pc.staub_problem()        # the six staub curves (nx = 128) and a measurement
    params = _capi.pack_params(bench.draw_states(4096, seed=20261018), bench.IDX, bench.UNITS)
    aux = _capi.default_aux(4096, 6, [1.0] * 6)
    kernels = (("warp", 0), ("cta", _capi.OPT_CTA_PER_TRAJ), ("seulex_warp", _capi.OPT_EXTRAPOLATION),
               ("seulex_cta", _capi.OPT_EXTRAPOLATION | _capi.OPT_CTA_PER_TRAJ))
    sizes = [1, 8, 32, 64, 128, 256, 1024, 4096]
else:
    from tests.test_extrapolation_traps import jittered_states, traps128_problem
    g, names, idx, prob = traps128_problem()
    params = _capi.pack_params(jittered_states(g, names, 4096, seed=1), idx, g["units"], model="traps")
    aux = _capi.default_aux(4096, 2, [1.0] * 2)
    kernels = (("warp", 0), ("seulex_cta", _capi.OPT_EXTRAPOLATION | _capi.OPT_CTA_PER_TRAJ))
    # 3 / 24 / 96 sets: the 6 / 48 / 192 trajectories of the staub rows (1 / 8 / 32 sets x 6 curves)
    sizes = [1, 3, 8, 24, 32, 96, 128, 256, 1024, 4096]
ctx.set_problem(prob)
out = []
for n in [int(a) for a in args] or sizes:
    row = {"n_sets": n, "n_traj": n * prob.n_meas}
    for name, flag in kernels:
        opts = _capi.make_opts(RTOL=1e-7, flags=flag | _capi.OPT_NO_EXPLICIT)
        ms = []
        for rep in range(6):
            ctx.upload(params[:n], aux[:n])
            ctx.run_resident(opts)
            ll, st, ns, _ = ctx.download()
            ms.append(ctx.last_kernel_ms())
        row[name + "_ms"] = float(np.median(ms[1:]))
        row[name + "_steps_max"] = int(ns.sum(axis=-1).max())
        row[name + "_steps_mean"] = float(ns.sum(axis=-1).mean())
    if "cta_ms" in row:
        row["speedup_cta"] = row["warp_ms"] / row["cta_ms"]
    row["speedup_seulex_cta"] = row["warp_ms"] / row["seulex_cta_ms"]
    out.append(row)
    print(json.dumps(row), flush=True)
