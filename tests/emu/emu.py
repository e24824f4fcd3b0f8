"""Loader for the host lock-step build of the kernel source (tests only)."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from metrotrpl_b200 import _capi

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "trpl_emu.cpp")
CSRC = os.path.join(HERE, "..", "..", "metrotrpl_b200", "csrc")
HEADER = os.path.join(HERE, "..", "..", "include", "metrotrpl_b200.h")
# team -> (library name, defines): one warp per trajectory, and the same source with the two-warp and
# the four-warp team vocabularies
VARIANTS = {0: ("libtrpl_emu", []), 2: ("libtrpl_emu_team", ["-DTRPL_TEAM=2"]),
            4: ("libtrpl_emu_team4", ["-DTRPL_TEAM=4"])}


def _deps():
    return [SRC, HEADER] + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".h")]


def build(force=False):
    """Compile the three variants next to the source; where the tree is read-only, into a temporary
    directory keyed by the sources.  Returns {team: path}."""
    deps = _deps()
    key = None
    if not os.access(HERE, os.W_OK):
        key = hashlib.sha1(b"".join(open(d, "rb").read() for d in sorted(deps))).hexdigest()[:16]
    paths = {}
    for team, (name, extra) in VARIANTS.items():
        so = os.path.join(HERE, f"{name}.so") if key is None else os.path.join(tempfile.gettempdir(), f"{name}_{key}.so")
        if force or not os.path.exists(so) or any(os.path.getmtime(so) < os.path.getmtime(d) for d in deps):
            tmp = f"{so}.{os.getpid()}.tmp"
            subprocess.check_call(["g++", "-std=c++17", "-O2", "-fopenmp", "-ffp-contract=off", "-shared",
                                   "-fPIC"] + extra + ["-o", tmp, SRC])
            os.replace(tmp, so)
        paths[team] = so
    return paths


_libs = {}


def lib(team=0):
    """The host lock-step build: one warp per trajectory (nx <= 128), the two-warp team (team=2, nx
    129..256) or the four-warp team (team=4, nx 257..512)."""
    team = int(team)
    if team not in _libs:
        l = C.CDLL(build()[team])
        dp, ip = C.POINTER(C.c_double), C.POINTER(C.c_int32)
        l.trpl_emu_loglik_batch.argtypes = [C.c_int32, C.c_int32, C.POINTER(_capi.MeasDesc), C.c_int32,
                                            dp, dp, dp, dp, C.c_int32, dp, dp,
                                            C.POINTER(_capi.SolverOpts), dp, ip, ip, dp, dp, dp, C.c_int32, dp, dp]
        l.trpl_emu_loglik_batch.restype = C.c_char_p
        _libs[team] = l
    return _libs[team]


def loglik_batch(prob, params, aux, opts, want_curves=True, ladder=None, fit=False):
    """(logll, status, nsteps, curves) of the host build, then the ladder rows [n_sets, n_meas, n_temps]
    when `ladder` (the temperatures) is given, then the fitted curves (TRPL_OPT_FIT) when `fit` is true.
    curves is None without want_curves.  The run stores what the library's run stores, whatever is
    returned."""
    params = np.ascontiguousarray(params, dtype=np.float64)
    aux = np.ascontiguousarray(aux, dtype=np.float64)
    n_sets = params.shape[0]
    logll = np.empty((n_sets, prob.n_meas, 3))
    status = np.empty((n_sets, prob.n_meas), dtype=np.int32)
    nsteps = np.empty((n_sets, prob.n_meas, 2), dtype=np.int32)
    curves = np.empty((n_sets, prob.n_times_total)) if want_curves else None
    p = _capi._ptr
    lad_T = None if ladder is None else np.ascontiguousarray(ladder, dtype=np.float64)
    lad_out = None if ladder is None else np.empty((n_sets, prob.n_meas, lad_T.size))
    fit_out = np.empty((n_sets, prob.n_times_total)) if fit else None
    if fit:
        opts = _capi.SolverOpts(opts.rtol, opts.atol, opts.hmax, opts.max_steps, opts.flags | _capi.OPT_FIT)
    # grids of more than 128 nodes run on the two-warp team, as in the product (the extrapolation
    # integrator's generic one-warp driver keeps its 8-nodes-per-lane host instantiation)
    max_nx = max(int(prob.meas[i].nx) for i in range(prob.n_meas))
    team = 0 if (max_nx <= 128 or (opts.flags & _capi.OPT_EXTRAPOLATION)) else (2 if max_nx <= 256 else 4)
    err = lib(team).trpl_emu_loglik_batch(prob.model, prob.n_meas, prob.meas, prob.n_times_total,
                                          p(prob.times, C.c_double), p(prob.vals, C.c_double),
                                          p(prob.uncs, C.c_double), p(prob.profiles, C.c_double), n_sets,
                                          p(params, C.c_double), p(aux, C.c_double), C.byref(opts),
                                          p(logll, C.c_double), p(status, C.c_int32), p(nsteps, C.c_int32),
                                          p(curves, C.c_double), p(prob.irf_moments, C.c_double),
                                          p(lad_T, C.c_double), 0 if ladder is None else lad_T.size,
                                          p(lad_out, C.c_double), p(fit_out, C.c_double))
    if err:
        raise RuntimeError(err.decode())
    return (logll, status, nsteps, curves) + (() if ladder is None else (lad_out,)) + ((fit_out,) if fit else ())
