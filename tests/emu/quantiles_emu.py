"""Loader for the host lock-step build of trpl_fit_quantiles (tests only): quantiles_emu.cpp runs the
selection routines of metrotrpl_b200/csrc/fit_quantiles.h on the host."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from metrotrpl_b200 import _capi

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "quantiles_emu.cpp")
CSRC = os.path.join(HERE, "..", "..", "metrotrpl_b200", "csrc")
DEPS = [SRC, os.path.join(HERE, "..", "..", "include", "metrotrpl_b200.h")] + \
       [os.path.join(CSRC, f) for f in ("fit_quantiles.h", "simt.h")]


def build():
    """Compile into the temporary directory, keyed by the sources (the tree may be read-only)."""
    key = hashlib.sha1(b"".join(open(d, "rb").read() for d in DEPS)).hexdigest()[:16]
    so = os.path.join(tempfile.gettempdir(), f"libtrpl_quantiles_emu_{key}.so")
    if not os.path.exists(so):
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
        dp, ip = C.POINTER(C.c_double), C.POINTER(C.c_int32)
        l.trpl_emu_fit_quantiles.argtypes = [C.c_int32, C.c_int32, dp, C.c_int32, dp, dp, ip]
        l.trpl_emu_fit_quantiles.restype = C.c_char_p
        _lib = l
    return _lib


def fit_quantiles(fit, q):
    """(quant [n_q, n_cols], count [n_cols]) of the host build's trpl_fit_quantiles on the fit buffer
    fit [n_sets, n_cols]; refusals raise ValueError with the library's message."""
    fit = np.ascontiguousarray(fit, dtype=np.float64)
    q = np.ascontiguousarray(np.atleast_1d(q), dtype=np.float64)
    n_sets, n_cols = fit.shape
    quant = np.empty((q.size, n_cols))
    count = np.empty(n_cols, dtype=np.int32)
    p = _capi._ptr
    err = lib().trpl_emu_fit_quantiles(n_sets, n_cols, p(fit, C.c_double), q.size, p(q, C.c_double),
                                       p(quant, C.c_double), p(count, C.c_int32))
    if err:
        raise ValueError(err.decode())
    return quant, count
