"""ctypes binding of include/metrotrpl_b200.h and the array packing both sides of it need.

No PyTorch, no CPU fallback: if the CUDA library is missing or no device is present,
:class:`Context` raises.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass, field
from typing import Optional, Sequence

import numpy as np

ABI_VERSION = 4
NPARAM = 16
NAUX = 6
NTEMP = 3

# parameter slots, include/metrotrpl_b200.h trpl_param_slot
PARAM_SLOTS = ("n0", "p0", "mu_n", "mu_p", "ks", "Cn", "Cp", "Sf", "Sb", "tauN", "tauP", "eps",
               "Tm", "kC", "Nt", "tauE")
TRAP_ONLY = ("kC", "Nt", "tauE")
A_SCALE_SHIFT, A_S2T0, A_S2T1, A_S2T2, A_FLUENCE_MULT, A_ABSORB_MULT = range(6)

MODEL_IDS = {"std": 0, "traps": 1}
MEAS_IDS = {"TRPL": 0, "TRTS": 1}
INI_IDS = {"density": 0, "fluence": 1}

ST_MAX_STEPS, ST_H_UNDERFLOW, ST_NONFINITE, ST_FLOORED, ST_NEG_FRAC, ST_NAN_LL, ST_CONV_FAIL = 1, 2, 4, 8, 16, 32, 64
ST_EXPLICIT = 128
OPT_FORCE_MIN_Y, OPT_NO_LIKELIHOOD, OPT_LADDER, OPT_NO_EXPLICIT, OPT_CTA_PER_TRAJ, OPT_EXTRAPOLATION = 1, 2, 4, 8, 16, 32
OPT_FIT = 64      # also keep the fitted curves (Context.download_fit)
MAX_QUANTILES = 8     # TRPL_MAX_QUANTILES: levels per Context.fit_quantiles call

# Defaults of the integrator.  RTOL keeps the reference's default value and meaning
# (forward_solver.py:18).  The reference's default ATOL (1e-10 nm^-3, forward_solver.py:19) is larger
# than the excess-carrier densities of low-injection curves; LSODA is only accurate there because
# of its hmax-limited steps, so a tolerance-proportional integrator must not honour it literally.
# See DESIGN.md "Tolerances".
DEFAULT_RTOL = 1e-7
ATOL_CEILING = 1e-30
DEFAULT_MAX_STEPS = 200000


class MeasDesc(C.Structure):
    _fields_ = [("thickness", C.c_double), ("ini_a", C.c_double), ("ini_b", C.c_double),
                ("nx", C.c_int32), ("meas_type", C.c_int32), ("ini_mode", C.c_int32),
                ("ini_dir", C.c_int32), ("n_t", C.c_int32), ("t_off", C.c_int32),
                ("prof_off", C.c_int32), ("irf_nk", C.c_int32), ("irf_dt", C.c_double),
                ("irf_off", C.c_int32), ("pad_", C.c_int32), ("min_y", C.c_double)]


class SolverOpts(C.Structure):
    _fields_ = [("rtol", C.c_double), ("atol", C.c_double), ("hmax", C.c_double),
                ("max_steps", C.c_int32), ("flags", C.c_int32)]


def check_extrapolation_problem(model, nx) -> None:
    """Raise ValueError unless the problem can run on the low-latency extrapolation integrator
    (OPT_EXTRAPOLATION, csrc/extrapolation.h): the 'std' or 'traps' model with nx = 128 on every
    measurement.  model: name as in MODEL_IDS; nx: nodes of each measurement."""
    if model not in ("std", "traps") or any(int(n) != 128 for n in nx):
        raise ValueError("kernel='seulex' needs the 'std' or 'traps' model with nx = 128 on every measurement")


def effective_tolerances(RTOL=None, ATOL=None):
    """Map the reference's (RTOL, ATOL) arguments onto the Rosenbrock controller."""
    rtol = DEFAULT_RTOL if RTOL is None else float(RTOL)
    atol = ATOL_CEILING if ATOL is None else min(float(ATOL), ATOL_CEILING)
    if not rtol > 0:
        raise ValueError("RTOL must be positive")
    return rtol, atol


def make_opts(RTOL=None, ATOL=None, hmax=0.0, honor_hmax=False, max_steps=DEFAULT_MAX_STEPS,
              flags=0) -> SolverOpts:
    rtol, atol = effective_tolerances(RTOL, ATOL)
    return SolverOpts(rtol, atol, float(hmax) if honor_hmax else 0.0, int(max_steps), int(flags))


@dataclass
class PackedProblem:
    """The measurement set in the flat layout trpl_set_problem takes."""
    model: int
    meas: np.ndarray            # array of MeasDesc (ctypes array)
    n_meas: int
    times: np.ndarray
    vals: Optional[np.ndarray]
    uncs: Optional[np.ndarray]
    profiles: Optional[np.ndarray]
    t_off: np.ndarray
    n_t: np.ndarray
    meas_types: list = field(default_factory=list)
    irf_moments: Optional[np.ndarray] = None     # [rows, 3] concatenated moment tables

    @property
    def n_times_total(self) -> int:
        return int(self.times.size)


def pack_problem(sim_info, init_params, times, vals=None, uncs=None, model="std",
                 ini_mode="density", irf_convolution=None, irf_tables=None, min_y=None) -> PackedProblem:
    """Flatten sim_info / _init_params / _times / _vals / _uncs (metropolis.py:317-326).

    irf_convolution : per-measurement wavelength (0 = none), shared_fields["irf_convolution"]
    irf_tables      : {wavelength: (moments[nk,3], t_irf)}, shared_fields["_IRF_tables"]
    """
    if model not in MODEL_IDS:
        raise ValueError(f"Invalid model {model}")
    if ini_mode not in INI_IDS:
        raise ValueError("Invalid ini_mode - must be 'density' or 'fluence'")
    n_meas = int(sim_info["num_meas"])
    descs = (MeasDesc * n_meas)()
    t_all, v_all, u_all, prof_all = [], [], [], []
    t_off = 0
    p_off = 0
    irf_rows = {}
    irf_blocks = []
    n_irf_rows = 0
    for i in range(n_meas):
        t = np.ascontiguousarray(times[i], dtype=np.float64)
        if t.ndim != 1 or t.size < 1:
            raise ValueError("each measurement needs a 1-D time array")
        if t[0] != 0:
            raise ValueError("Grid error - times must start at t=0")      # sim_utils.py:271-272
        mtype = sim_info["meas_types"][i]
        if mtype not in MEAS_IDS:
            raise NotImplementedError("TRTS or TRPL only")               # forward_solver.py:202-203
        nx = int(sim_info["nx"][i])
        ini = np.asarray(init_params[i], dtype=np.float64)
        d = descs[i]
        d.thickness = float(sim_info["lengths"][i])
        d.nx = nx
        d.meas_type = MEAS_IDS[mtype]
        d.ini_mode = INI_IDS[ini_mode]
        d.n_t = t.size
        d.t_off = t_off
        d.ini_dir = 1
        d.min_y = float(np.finfo(float).tiny if min_y is None else min_y[i])   # Grid.min_y, sim_utils.py:281
        if ini_mode == "density":
            if ini.size != nx:                                            # forward_solver.py:101-104
                raise ValueError(
                    f"Expected {nx} initial densities but initial condition file has {ini.size}")
            d.prof_off = p_off
            prof_all.append(ini)
            p_off += nx
        else:
            if ini.size > 3:                                              # forward_solver.py:106-115
                raise ValueError("Expected only fluence, absorption coef, and direction but "
                                 f"initial condition file has {ini.size} values")
            d.ini_a = float(ini[0])
            d.ini_b = float(ini[1])
            try:
                d.ini_dir = int(np.sign(int(ini[2]))) or 1                # sign 0 -> slice error -> unchanged
            except (IndexError, ValueError):
                d.ini_dir = 1
        if irf_convolution is not None and irf_convolution[i] != 0:
            wave = int(irf_convolution[i])
            mom, t_irf = irf_tables[wave]
            if wave not in irf_rows:
                irf_rows[wave] = n_irf_rows
                irf_blocks.append(np.ascontiguousarray(mom, dtype=np.float64))
                n_irf_rows += len(mom)
            d.irf_off = irf_rows[wave]
            d.irf_nk = len(mom)
            d.irf_dt = float(np.mean(np.diff(t_irf)))                   # laplace.py:66
        t_all.append(t)
        if vals is not None:
            v = np.ascontiguousarray(vals[i], dtype=np.float64)
            u = np.ascontiguousarray(uncs[i], dtype=np.float64)
            if v.size != t.size or u.size != t.size:
                raise ValueError("times / vals / uncs length mismatch")
            v_all.append(v)
            u_all.append(u)
        t_off += t.size
    return PackedProblem(
        model=MODEL_IDS[model], meas=descs, n_meas=n_meas,
        times=np.concatenate(t_all),
        vals=np.concatenate(v_all) if vals is not None else None,
        uncs=np.concatenate(u_all) if vals is not None else None,
        profiles=np.concatenate(prof_all) if prof_all else None,
        t_off=np.array([d.t_off for d in descs], dtype=np.int64),
        n_t=np.array([d.n_t for d in descs], dtype=np.int64),
        meas_types=list(sim_info["meas_types"]),
        irf_moments=np.concatenate(irf_blocks) if irf_blocks else None)


def pack_params(states, indexes, units=None, model="std") -> np.ndarray:
    """[n_sets, n_names] states in file units -> [n_sets, NPARAM] model-unit rows.

    Mirrors forward_solver.py:119-138: state * units, then pick by name.
    """
    states = np.atleast_2d(np.asarray(states, dtype=np.float64))
    if units is None:
        units = np.ones(states.shape[1])
    conv = states * np.asarray(units, dtype=np.float64)[None, :]
    out = np.zeros((states.shape[0], NPARAM))
    for slot, name in enumerate(PARAM_SLOTS):
        if name in TRAP_ONLY and model != "traps":
            out[:, slot] = 1.0 if name == "tauE" else 0.0
            continue
        if name not in indexes:
            raise KeyError(name)
        out[:, slot] = conv[:, indexes[name]]
    return np.ascontiguousarray(out)


def _ptr(a, ctype):
    if a is None:
        return None
    return a.ctypes.data_as(C.POINTER(ctype))


_LIB_NAME = "libmetrotrpl_b200.so"


def library_path() -> str:
    # METROTRPL_B200_LIB: developer override to A/B another build of the same CUDA library
    override = os.environ.get("METROTRPL_B200_LIB")
    if override:
        return os.path.abspath(override)
    return os.path.join(os.path.dirname(os.path.abspath(__file__)), _LIB_NAME)


def load_library() -> C.CDLL:
    path = library_path()
    if not os.path.exists(path):
        raise RuntimeError(
            f"{path} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'`. "
            "metrotrpl_b200 has no CPU fallback.")
    lib = C.CDLL(path)
    dp, ip = C.POINTER(C.c_double), C.POINTER(C.c_int32)
    H = C.c_void_p
    lib.trpl_last_error.restype = C.c_char_p
    lib.trpl_abi_version.restype = C.c_int
    lib.trpl_create.argtypes = [C.c_int, C.POINTER(H)]
    lib.trpl_destroy.argtypes = [H]
    lib.trpl_destroy.restype = None
    lib.trpl_device_info.argtypes = [H, ip, ip, C.c_char_p, C.c_int32]
    lib.trpl_set_problem.argtypes = [H, C.c_int32, C.c_int32, C.POINTER(MeasDesc), C.c_int32, dp, dp,
                                     dp, C.c_int32, dp]
    lib.trpl_set_irf.argtypes = [H, C.c_int32, dp]
    lib.trpl_set_ladder.argtypes = [H, C.c_int32, dp]
    lib.trpl_download_ladder.argtypes = [H, dp]
    lib.trpl_download_ladder_sums.argtypes = [H, dp, ip]
    lib.trpl_ladder_sums_resident.argtypes = [H, C.POINTER(C.c_void_p), ip, ip]
    lib.trpl_download_nsteps.argtypes = [H, ip]
    lib.trpl_loglik_batch.argtypes = [H, C.c_int32, dp, dp, C.POINTER(SolverOpts), dp, ip, ip, dp]
    lib.trpl_solve_batch.argtypes = [H, C.c_int32, dp, dp, C.POINTER(SolverOpts), dp, ip, ip]
    lib.trpl_upload_batch.argtypes = [H, C.c_int32, dp, dp]
    lib.trpl_run_resident.argtypes = [H, C.POINTER(SolverOpts), C.c_int32]
    lib.trpl_download_results.argtypes = [H, dp, ip, ip, dp]
    lib.trpl_download_fit.argtypes = [H, dp]
    lib.trpl_fit_quantiles.argtypes = [H, C.c_int32, dp, dp, ip]
    lib.trpl_last_kernel_ms.argtypes = [H, C.POINTER(C.c_float)]
    lib.trpl_launch_count.argtypes = [H]
    lib.trpl_launch_count.restype = C.c_int64
    u8p, u64p, u32p = C.POINTER(C.c_uint8), C.POINTER(C.c_uint64), C.POINTER(C.c_uint32)
    lib.trpl_make_trial_moves.argtypes = [C.c_int32, C.c_int32, dp, dp, u8p, u8p, dp, dp, C.c_int32, C.c_int32,
                                          C.c_int32, C.c_int32, C.c_int32, C.c_int32, u64p, u64p, dp, dp,
                                          C.POINTER(C.c_int64), ip, u32p, C.c_int32, C.c_int32, C.c_double,
                                          C.c_double, dp, C.c_int32, ip, dp]
    lib.trpl_set_queue_order.argtypes = [H, C.c_int32, ip]
    lib.trpl_synchronize.argtypes = [H]
    lib.trpl_timer_begin.argtypes = [H]
    lib.trpl_timer_end.argtypes = [H, C.POINTER(C.c_float)]
    lib.trpl_flush_l2.argtypes = [H]
    lib.trpl_fp64_peak_probe.argtypes = [H, C.c_int32, dp, C.POINTER(C.c_float)]
    return lib


class TrplError(RuntimeError):
    pass


class Context:
    """One CUDA device, one measurement set at a time (one process per GPU)."""

    def __init__(self, device: int = 0):
        self.lib = load_library()
        if self.lib.trpl_abi_version() != ABI_VERSION:
            raise TrplError("ABI version mismatch")
        self.h = C.c_void_p()
        self._check(self.lib.trpl_create(int(device), C.byref(self.h)))
        self.problem: Optional[PackedProblem] = None
        self.device = int(device)

    def _check(self, rc):
        if rc != 0:
            raise TrplError(self.lib.trpl_last_error().decode())

    def close(self):
        if getattr(self, "h", None) is not None and self.h:
            self.lib.trpl_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    def device_info(self):
        sm, khz = C.c_int32(), C.c_int32()
        name = C.create_string_buffer(128)
        self._check(self.lib.trpl_device_info(self.h, C.byref(sm), C.byref(khz), name, 128))
        return {"sm_count": sm.value, "sm_clock_khz": khz.value, "name": name.value.decode()}

    def set_problem(self, prob: PackedProblem):
        nprof = 0 if prob.profiles is None else int(prob.profiles.size)
        self._check(self.lib.trpl_set_problem(
            self.h, prob.model, prob.n_meas, prob.meas, prob.n_times_total,
            _ptr(prob.times, C.c_double), _ptr(prob.vals, C.c_double), _ptr(prob.uncs, C.c_double),
            nprof, _ptr(prob.profiles, C.c_double)))
        if prob.irf_moments is not None:
            self._check(self.lib.trpl_set_irf(self.h, int(prob.irf_moments.shape[0]),
                                              _ptr(prob.irf_moments, C.c_double)))
        self.problem = prob

    def set_problem_if_needed(self, prob: PackedProblem):
        if self.problem is not prob:
            self.set_problem(prob)

    def set_queue_order(self, order=None):
        """Order in which the persistent warps claim trajectories (index = set * n_meas + meas) in the
        next launches of exactly len(order) trajectories; None restores the built-in order."""
        if order is None:
            self._check(self.lib.trpl_set_queue_order(self.h, 0, None))
            return
        order = np.ascontiguousarray(order, dtype=np.int32)
        self._check(self.lib.trpl_set_queue_order(self.h, int(order.size), _ptr(order, C.c_int32)))

    def set_ladder(self, temps):
        temps = np.ascontiguousarray(temps, dtype=np.float64)
        self._check(self.lib.trpl_set_ladder(self.h, temps.size, _ptr(temps, C.c_double)))
        self._n_ladder = temps.size

    def download_ladder(self, n_sets):
        out = np.empty((n_sets, self.problem.n_meas, self._n_ladder))
        self._check(self.lib.trpl_download_ladder(self.h, _ptr(out, C.c_double)))
        return out

    def download_ladder_sums(self, n_sets, want_nsteps=True):
        """[n_sets, n_temps] per-chain likelihood at every ladder temperature (summed over the
        measurements, NaN -> -inf) and the step counts, one synchronisation."""
        rows = np.empty((n_sets, self._n_ladder))
        nsteps = np.empty((n_sets, self.problem.n_meas, 2), dtype=np.int32) if want_nsteps else None
        self._check(self.lib.trpl_download_ladder_sums(self.h, _ptr(rows, C.c_double), _ptr(nsteps, C.c_int32)))
        return rows, nsteps

    def ladder_sums_resident(self):
        """(device pointer, n_sets, n_temps) of the same rows, left in HBM (stream synchronised)."""
        ptr = C.c_void_p()
        n, k = C.c_int32(), C.c_int32()
        self._check(self.lib.trpl_ladder_sums_resident(self.h, C.byref(ptr), C.byref(n), C.byref(k)))
        return ptr.value, n.value, k.value

    def download_nsteps(self, n_sets):
        nsteps = np.empty((n_sets, self.problem.n_meas, 2), dtype=np.int32)
        self._check(self.lib.trpl_download_nsteps(self.h, _ptr(nsteps, C.c_int32)))
        return nsteps

    # -- whole-batch calls (host buffers in, host buffers out) --
    def loglik_batch(self, params, aux, opts: SolverOpts, want_curves=False):
        prob = self.problem
        params = np.ascontiguousarray(params, dtype=np.float64)
        aux = np.ascontiguousarray(aux, dtype=np.float64)
        n_sets = params.shape[0]
        n_traj = n_sets * prob.n_meas
        assert params.shape == (n_sets, NPARAM) and aux.size == n_traj * NAUX
        logll = np.empty((n_sets, prob.n_meas, NTEMP))
        status = np.empty((n_sets, prob.n_meas), dtype=np.int32)
        nsteps = np.empty((n_sets, prob.n_meas, 2), dtype=np.int32)
        curves = np.empty((n_sets, prob.n_times_total)) if want_curves else None
        self._n_sets = n_sets
        self._check(self.lib.trpl_loglik_batch(
            self.h, n_sets, _ptr(params, C.c_double), _ptr(aux, C.c_double), C.byref(opts),
            _ptr(logll, C.c_double), _ptr(status, C.c_int32), _ptr(nsteps, C.c_int32),
            _ptr(curves, C.c_double)))
        return logll, status, nsteps, curves

    def solve_batch(self, params, aux, opts: SolverOpts):
        prob = self.problem
        params = np.ascontiguousarray(params, dtype=np.float64)
        aux = np.ascontiguousarray(aux, dtype=np.float64)
        n_sets = params.shape[0]
        status = np.empty((n_sets, prob.n_meas), dtype=np.int32)
        nsteps = np.empty((n_sets, prob.n_meas, 2), dtype=np.int32)
        curves = np.empty((n_sets, prob.n_times_total))
        self._check(self.lib.trpl_solve_batch(
            self.h, n_sets, _ptr(params, C.c_double), _ptr(aux, C.c_double), C.byref(opts),
            _ptr(curves, C.c_double), _ptr(status, C.c_int32), _ptr(nsteps, C.c_int32)))
        return curves, status, nsteps

    # -- split calls for device-resident timing --
    def upload(self, params, aux):
        params = np.ascontiguousarray(params, dtype=np.float64)
        aux = np.ascontiguousarray(aux, dtype=np.float64)
        self._n_sets = params.shape[0]
        self._check(self.lib.trpl_upload_batch(self.h, params.shape[0], _ptr(params, C.c_double),
                                               _ptr(aux, C.c_double)))

    def run_resident(self, opts: SolverOpts, want_curves=False):
        self._check(self.lib.trpl_run_resident(self.h, C.byref(opts), 1 if want_curves else 0))

    def download(self, want_curves=False):
        prob = self.problem
        n_sets = self._n_sets
        logll = np.empty((n_sets, prob.n_meas, NTEMP))
        status = np.empty((n_sets, prob.n_meas), dtype=np.int32)
        nsteps = np.empty((n_sets, prob.n_meas, 2), dtype=np.int32)
        curves = np.empty((n_sets, prob.n_times_total)) if want_curves else None
        self._check(self.lib.trpl_download_results(
            self.h, _ptr(logll, C.c_double), _ptr(status, C.c_int32), _ptr(nsteps, C.c_int32),
            _ptr(curves, C.c_double)))
        return logll, status, nsteps, curves

    def download_fit(self):
        """[n_sets, n_times_total] fitted curves of the last run, which had OPT_FIT: per point what the
        likelihood compared with vals, log10(|signal|) + log10(_s#) after the min_y floor and, with an
        IRF, after convolution and trim; NaN past the compared points (include/metrotrpl_b200.h,
        trpl_download_fit)."""
        fit = np.empty((self._n_sets, self.problem.n_times_total))
        self._check(self.lib.trpl_download_fit(self.h, _ptr(fit, C.c_double)))
        return fit

    def fit_quantiles(self, q):
        """(quant [n_q, n_times_total], count [n_times_total]) over the parameter sets of the last run,
        which had OPT_FIT: quant equals np.nanquantile(download_fit(), q, axis=0, method="linear") bit
        for bit, count the sets whose fitted point is not NaN.  The selection runs on the device; only
        these two arrays are copied to the host (include/metrotrpl_b200.h, trpl_fit_quantiles)."""
        q = np.ascontiguousarray(np.atleast_1d(q), dtype=np.float64)
        n = self.problem.n_times_total
        quant = np.empty((q.size, n))
        count = np.empty(n, dtype=np.int32)
        self._check(self.lib.trpl_fit_quantiles(self.h, int(q.size), _ptr(q, C.c_double), _ptr(quant, C.c_double),
                                                _ptr(count, C.c_int32)))
        return quant, count

    def last_kernel_ms(self) -> float:
        ms = C.c_float()
        self._check(self.lib.trpl_last_kernel_ms(self.h, C.byref(ms)))
        return float(ms.value)

    def launch_count(self) -> int:
        return int(self.lib.trpl_launch_count(self.h))

    def synchronize(self):
        self._check(self.lib.trpl_synchronize(self.h))

    def timer_begin(self):
        self._check(self.lib.trpl_timer_begin(self.h))

    def timer_end(self) -> float:
        ms = C.c_float()
        self._check(self.lib.trpl_timer_end(self.h, C.byref(ms)))
        return float(ms.value)

    def flush_l2(self):
        self._check(self.lib.trpl_flush_l2(self.h))

    def fp64_peak_probe(self, iters=20000):
        tf = C.c_double()
        ms = C.c_float()
        self._check(self.lib.trpl_fp64_peak_probe(self.h, int(iters), C.byref(tf), C.byref(ms)))
        return float(tf.value), float(ms.value)


def default_aux(n_sets, n_meas, sigma_by_meas: Sequence[float], temps=(1.0, 1.0, 1.0),
                scale_shift=0.0, fl_mult=1.0, al_mult=1.0) -> np.ndarray:
    """aux rows for the plain case: per-measurement model uncertainty, up to three temperatures."""
    aux = np.zeros((n_sets, n_meas, NAUX))
    aux[..., A_SCALE_SHIFT] = scale_shift
    s2 = np.asarray(sigma_by_meas, dtype=np.float64) ** 2
    temps = np.broadcast_to(np.asarray(temps, dtype=np.float64), (n_sets, 3)) if np.ndim(temps) < 2 \
        else np.asarray(temps, dtype=np.float64)
    for k in range(3):
        aux[..., A_S2T0 + k] = s2[None, :] * temps[:, k][:, None]
    aux[..., A_FLUENCE_MULT] = fl_mult
    aux[..., A_ABSORB_MULT] = al_mult
    return aux
