"""Loader for the host lock-step build of the fitted-curve pass (tests only): the library's
TRPL_OPT_FIT pass (trajectory.h fit_trajectory) run on the curves of the host lock-step build."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from metrotrpl_b200 import _capi
from tests.emu import emu

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "trpl_emu_fit.cpp")
SO = os.path.join(HERE, "libtrpl_emu_fit.so")


def _deps():
    return [SRC] + [os.path.join(emu.CSRC, f) for f in os.listdir(emu.CSRC) if f.endswith(".h")]


def build(force=False):
    """Compile next to the source; where the tree is read-only, into a temporary directory keyed by
    the sources."""
    so = SO
    if not os.access(HERE, os.W_OK):
        h = hashlib.sha1(b"".join(open(d, "rb").read() for d in sorted(_deps()))).hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), f"libtrpl_emu_fit_{h}.so")
    if force or not os.path.exists(so) or any(os.path.getmtime(so) < os.path.getmtime(d) for d in _deps()):
        tmp = f"{so}.{os.getpid()}.tmp"
        subprocess.check_call(["g++", "-std=c++17", "-O2", "-fopenmp", "-ffp-contract=off", "-shared", "-fPIC",
                               "-o", tmp, SRC])
        os.replace(tmp, so)
    return so


_lib = None


def lib():
    global _lib
    if _lib is None:
        l = C.CDLL(build())
        dp = C.POINTER(C.c_double)
        l.trpl_emu_fit_batch.argtypes = [C.c_int32, C.POINTER(_capi.MeasDesc), C.c_int32, dp, dp, dp, C.c_int32,
                                         dp, C.POINTER(_capi.SolverOpts), dp, dp, dp]
        _lib = l
    return _lib


def fit_batch(prob, aux, opts, curves):
    """[n_sets, n_times_total] fitted curves of a run from its curves, as TRPL_OPT_FIT computes them."""
    aux = np.ascontiguousarray(aux, dtype=np.float64)
    curves = np.ascontiguousarray(curves, dtype=np.float64)
    n_sets = curves.shape[0]
    assert curves.shape == (n_sets, prob.n_times_total) and aux.size == n_sets * prob.n_meas * _capi.NAUX
    fit = np.empty((n_sets, prob.n_times_total))
    p = _capi._ptr
    rc = lib().trpl_emu_fit_batch(prob.n_meas, prob.meas, prob.n_times_total, p(prob.times, C.c_double),
                                  p(prob.vals, C.c_double), p(prob.uncs, C.c_double), n_sets, p(aux, C.c_double),
                                  C.byref(opts), p(curves, C.c_double), p(prob.irf_moments, C.c_double),
                                  p(fit, C.c_double))
    if rc:
        raise RuntimeError("emu fit failed")
    return fit


def loglik_batch(prob, params, aux, opts, ladder=None):
    """emu.loglik_batch with the curves, plus the fitted curves: (logll, status, nsteps, curves, fit)."""
    res = emu.loglik_batch(prob, params, aux, opts, True, ladder=ladder)
    return (*res[:4], fit_batch(prob, aux, opts, res[3]))
