/* metrotrpl_b200.h - C ABI of the B200 forward-simulation + likelihood library.
 *
 * This is the drop-in boundary for MetroTRPL's data-parallel hot path.  The reference is pure
 * Python; the binding a maintainer adds is a ctypes stub (shown in INTEGRATION.md) that replaces
 *
 *   forward_solver.py:41-203        solve(iniPar, g, state, indexes, meas, units, solver, model,
 *                                         ini_mode, RTOL, ATOL)          -> trpl_solve_batch
 *   trial_move_evaluation.py:9-28   eval_trial_move(state, unique_fields, shared_fields, logger)
 *   trial_move_evaluation.py:30-166 one_sim_likelihood(...)             -> trpl_loglik_batch
 *   Dense_Sample/dense_sampling.py:42-196 simulate(...) inner loops      -> trpl_loglik_batch
 *   trial_move_generation.py:54-96 make_trial_move + metropolis.py:118-127 draw order
 *                                                                       -> trpl_make_trial_moves
 *
 * with whole batches of parameter sets per call instead of one state at a time.
 * Plain pointers and sizes only; all arrays are C-contiguous float64 / int32 HOST arrays unless a
 * function name says "resident".  Every function returns 0 on success, non-zero on failure;
 * trpl_last_error() returns a description.  There is no CPU fallback: without a CUDA device
 * trpl_create fails.
 */
#ifndef METROTRPL_B200_H
#define METROTRPL_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TRPL_ABI_VERSION 4
#define TRPL_NPARAM 16  /* doubles per parameter set, model units (nm, ns, V) */
#define TRPL_NAUX 6     /* doubles per trajectory, see below */
#define TRPL_NTEMP 3    /* likelihoods are returned for three temperatures per trajectory */

/* parameter slots (forward_solver.py:128-138 order; state[indexes[name]] * units) */
enum trpl_param_slot {
  TRPL_P_N0 = 0, TRPL_P_P0, TRPL_P_MUN, TRPL_P_MUP, TRPL_P_KS, TRPL_P_CN, TRPL_P_CP, TRPL_P_SF,
  TRPL_P_SB, TRPL_P_TAUN, TRPL_P_TAUP, TRPL_P_EPS, TRPL_P_TM, TRPL_P_KC, TRPL_P_NT, TRPL_P_TAUE
};
/* aux slots, one row per (parameter set, measurement) trajectory */
enum trpl_aux_slot {
  TRPL_A_SCALE_SHIFT = 0, /* log10(_s#), trial_move_evaluation.py:52-60 */
  TRPL_A_S2T0, TRPL_A_S2T1, TRPL_A_S2T2, /* model_uncertainty[meas_type]^2 * T, :150-156 */
  TRPL_A_FLUENCE_MULT, /* _f# factor, :38-44 */
  TRPL_A_ABSORB_MULT   /* _a# factor, :45-51 */
};

enum trpl_model { TRPL_MODEL_STD = 0, TRPL_MODEL_TRAPS = 1 };       /* forward_solver.py:420-423 */
enum trpl_meas_type { TRPL_MEAS_TRPL = 0, TRPL_MEAS_TRTS = 1 };      /* forward_solver.py:186-203 */
enum trpl_ini_mode { TRPL_INI_DENSITY = 0, TRPL_INI_FLUENCE = 1 };   /* forward_solver.py:100-117 */

/* status bits per trajectory */
enum trpl_status {
  TRPL_ST_OK = 0, TRPL_ST_MAX_STEPS = 1, TRPL_ST_H_UNDERFLOW = 2, TRPL_ST_NONFINITE = 4,
  TRPL_ST_FLOORED = 8, TRPL_ST_NEG_FRAC = 16, TRPL_ST_NAN_LL = 32, TRPL_ST_CONV_FAIL = 64,
  TRPL_ST_EXPLICIT = 128 /* informational: non-stiff trajectory, integrated by the explicit RK path */
};
enum trpl_opt_flags { TRPL_OPT_FORCE_MIN_Y = 1, TRPL_OPT_NO_LIKELIHOOD = 2, TRPL_OPT_LADDER = 4,
                      TRPL_OPT_NO_EXPLICIT = 8, /* always use the Rosenbrock integrator */
                      TRPL_OPT_CTA_PER_TRAJ = 16, /* one trajectory per CTA of 128 threads instead of one per
                                                    warp: lowest latency per trajectory, for small batches
                                                    (tempering); 'std' model, nx = 128 only */
                      TRPL_OPT_EXTRAPOLATION = 32, /* integrate with the order-6 extrapolation method
                                                    (csrc/extrapolation.h) instead of RODAS4; together with
                                                    TRPL_OPT_CTA_PER_TRAJ its six columns run in parallel on
                                                    the four warps of a CTA: a quarter of the latency per
                                                    trajectory; 'std' and 'traps' models, nx = 128 only */
                      TRPL_OPT_FIT = 64 /* also keep the fitted curves: what the likelihood compares, per
                                          point; see trpl_download_fit */ };

/* one measurement (sim_info["lengths"/"nx"/"meas_types"][i] + its slice of the data arrays) */
typedef struct trpl_meas_desc {
  double thickness;   /* nm */
  double ini_a;       /* fluence mode: fluence [cm^-2] */
  double ini_b;       /* fluence mode: absorption coefficient [cm^-1] */
  int32_t nx;         /* space nodes, 2..512 */
  int32_t meas_type;  /* trpl_meas_type */
  int32_t ini_mode;   /* trpl_ini_mode */
  int32_t ini_dir;    /* fluence mode: <0 reverses the profile */
  int32_t n_t;        /* measurement times of this curve; times[t_off] must be 0 */
  int32_t t_off;      /* offset into times / vals / uncs / per-set curves */
  int32_t prof_off;   /* density mode: offset into profiles (cm^-3, nx values) */
  int32_t irf_nk;     /* rows of this curve's IRF moment table (laplace.py:13-41); 0 = no convolution */
  double irf_dt;      /* mean IRF time step [ns] (laplace.py:66) */
  int32_t irf_off;    /* first row of the table in the array given to trpl_set_irf */
  int32_t pad_;
  double min_y;       /* signal floor, Grid.min_y (sim_utils.py:281; forward_solver.py:190-192) */
} trpl_meas_desc;

typedef struct trpl_solver_opts {
  double rtol;        /* relative local tolerance of the Rosenbrock controller (reference RTOL) */
  double atol;        /* absolute floor [nm^-3]; see DESIGN.md "tolerances" */
  double hmax;        /* > 0: cap on the step size [ns] (reference "hmax"); <= 0: error control only */
  int32_t max_steps;  /* accepted + rejected step budget per trajectory */
  int32_t flags;      /* trpl_opt_flags */
} trpl_solver_opts;

typedef struct trpl_handle trpl_handle;

const char* trpl_last_error(void);
int trpl_abi_version(void);

/* Create / destroy a context bound to one CUDA device (one process per GPU). */
int trpl_create(int device, trpl_handle** out);
void trpl_destroy(trpl_handle* h);
int trpl_device_info(trpl_handle* h, int32_t* sm_count, int32_t* sm_clock_khz, char* name, int32_t name_len);

/* Upload the measurement set shared by every parameter set of later calls
 * (shared_fields["_sim_info"], "_times", "_vals", "_uncs", "_init_params").  vals/uncs may be NULL
 * when only curves are wanted; profiles may be NULL in fluence mode. */
int trpl_set_problem(trpl_handle* h, int32_t model, int32_t n_meas, const trpl_meas_desc* meas,
                     int32_t n_times_total, const double* times, const double* vals,
                     const double* uncs, int32_t n_profile_total, const double* profiles);

/* IRF moment tables of every wavelength in use, rows of {I^0, I^1, I^2} concatenated
 * (shared_fields["_IRF_tables"], laplace.py:13-41).  Call after trpl_set_problem when any
 * measurement has irf_nk > 0; the in-kernel convolution replaces laplace.py:44-129. */
int trpl_set_irf(trpl_handle* h, int32_t n_rows_total, const double* moments);

/* Parallel-tempering ladder: with TRPL_OPT_LADDER every trajectory also returns its likelihood at
 * each of these temperatures (the reference's ll_func(T), trial_move_evaluation.py:150-156), so the
 * swap move (metropolis.py:66-90) needs no re-simulation.  aux slot TRPL_A_S2T1 must then hold
 * model_uncertainty^2 (temperature 1).  Results: trpl_download_ladder, [n_sets][n_meas][n_temps]. */
int trpl_set_ladder(trpl_handle* h, int32_t n_temps, const double* temps);
int trpl_download_ladder(trpl_handle* h, double* out);
/* The swap move only needs the sum over measurements (metropolis.py:73-76): rows [n_sets][n_temps],
 * NaN -> -inf.  trpl_download_ladder_sums copies them (and, if nsteps != NULL, the step counts
 * [n_sets][n_meas][2]) to the host with one stream synchronisation.  trpl_ladder_sums_resident leaves
 * them in HBM and returns the device pointer (valid until the next run on this handle; the stream is
 * synchronised, so a collective on another stream may read it): the rows of several GPUs are then
 * all-gathered device to device (NCCL) without touching the host. */
int trpl_download_ladder_sums(trpl_handle* h, double* rows, int32_t* nsteps);
int trpl_ladder_sums_resident(trpl_handle* h, const double** dev_rows, int32_t* n_sets, int32_t* n_temps);
int trpl_download_nsteps(trpl_handle* h, int32_t* nsteps);

/* Whole-batch likelihood: n_sets parameter sets x n_meas measurements.
 *   params  [n_sets][TRPL_NPARAM]
 *   aux     [n_sets][n_meas][TRPL_NAUX]
 *   logll   [n_sets][n_meas][TRPL_NTEMP]  per-curve log-likelihood (sum over n_meas = eval_trial_move)
 *   status  [n_sets][n_meas]              trpl_status bits
 *   nsteps  [n_sets][n_meas][2]           accepted, rejected steps (may be NULL)
 *   curves  [n_sets][n_times_total]       simulated signals in measurement units (may be NULL)
 * Host buffers in, host buffers out; H2D and D2H copies happen inside the call. */
int trpl_loglik_batch(trpl_handle* h, int32_t n_sets, const double* params, const double* aux,
                      const trpl_solver_opts* opts, double* logll, int32_t* status, int32_t* nsteps,
                      double* curves);

/* forward_solver.solve() for a batch: curves only (flags |= TRPL_OPT_NO_LIKELIHOOD). */
int trpl_solve_batch(trpl_handle* h, int32_t n_sets, const double* params, const double* aux,
                     const trpl_solver_opts* opts, double* curves, int32_t* status, int32_t* nsteps);

/* Fitted curves of the last run, which must have had TRPL_OPT_FIT (with the likelihood and uploaded
 * vals): fit [n_sets][n_times_total], laid out like curves.  For the trajectory (set s, measurement m),
 * point k < n_c holds log10(|y_k|) + scale_shift, the left operand of the likelihood's residual
 * r_k = fit_k - vals_k: y is the simulated signal after the min_y floor (and the TRPL_OPT_FORCE_MIN_Y
 * floor) or, for a measurement with an IRF, the convolved, max-shifted signal interpolated back onto
 * the measurement times.  n_c = n_t without IRF; with IRF it is the prefix of times inside the
 * convolved span.  Points k >= n_c are NaN, and so is the whole slice when the convolution failed
 * (TRPL_ST_CONV_FAIL).  The fit does not depend on the temperatures or model uncertainties in aux, and
 * asking for it changes no other output. */
int trpl_download_fit(trpl_handle* h, double* fit);

/* Per-point quantiles over the parameter sets of the last run, which must have had TRPL_OPT_FIT.
 *   q      [n_q] in [0, 1], 1 <= n_q <= TRPL_MAX_QUANTILES
 *   quant  [n_q][n_times_total]: np.nanquantile(fit, q, axis=0, method="linear"), bit for bit
 *   count  [n_times_total]: sets whose fitted point is not NaN (may be NULL)
 * Only quant and count are copied to the host; the fit buffer is not.  A point no set compared
 * (count 0) has NaN quantiles.  The fit buffer and every other result of the run stay as they are. */
#define TRPL_MAX_QUANTILES 8
int trpl_fit_quantiles(trpl_handle* h, int32_t n_q, const double* q, double* quant, int32_t* count);

/* Split form used for device-resident timing: inputs stay in HBM between runs. */
int trpl_upload_batch(trpl_handle* h, int32_t n_sets, const double* params, const double* aux);
int trpl_run_resident(trpl_handle* h, const trpl_solver_opts* opts, int32_t want_curves);
int trpl_download_results(trpl_handle* h, double* logll, int32_t* status, int32_t* nsteps, double* curves);
/* Duration of the last trajectory-kernel launch, CUDA events on the library's stream [ms]. */
int trpl_last_kernel_ms(trpl_handle* h, float* ms);
/* Number of kernel launches this context has issued (bench.py's gpu_launches claim). */
int64_t trpl_launch_count(trpl_handle* h);
int trpl_synchronize(trpl_handle* h);

/* Bracket a timed region with CUDA events on the library's stream (bench.py: K steps). */
int trpl_timer_begin(trpl_handle* h);
int trpl_timer_end(trpl_handle* h, float* ms);
/* Write a 256 MiB scratch buffer on the library's stream (evicts the 126 MB L2 between steps). */
int trpl_flush_l2(trpl_handle* h);

/* Queue order of the next launches: order[q] = index (set * n_meas + meas) of the q-th trajectory
 * the persistent warps claim.  Any permutation of [0, n_traj) is valid and none changes a result;
 * longest first shortens the tail of a launch (a Metropolis driver passes the step counts of the
 * previous iteration's proposals, sorted descending).  Applies to launches with exactly n_traj
 * trajectories until replaced; n_traj = 0 or order = NULL restores the built-in order
 * (measurement-major, statically most expensive curves first).  trpl_set_problem clears it. */
int trpl_set_queue_order(trpl_handle* h, int32_t n_traj, const int32_t* order);

/* Dependent-free DFMA stream on every SM: measured FP64 peak for the roofline denominator. */
int trpl_fp64_peak_probe(trpl_handle* h, int32_t iters, double* tflops, float* ms);

/* Host side of one Metropolis iteration: the proposals of ALL chains and their acceptance draws,
 * consuming a PCG64 stream (NumPy's default_rng) in exactly the order of the reference's serial
 * loop - for each chain in turn one draw per parameter and attempt (trial_move_generation.py:54-96,
 * retried up to max_tries times under hard bounds, checks of :4-52), then the chain's acceptance
 * draw (metropolis.py:118-127).  No device work.
 *   cur, moves        [n_chains][n_par] current states and box half-widths in the sampler's scale
 *                     (log10 of the parameters with do_log set); proposals come back in that scale
 *   do_log, active    [n_par] flags; lo, hi [n_par] prior bounds (linear units)
 *   idx_*             parameter indices of p0/n0 and tauN/tauP, or -1 when absent
 *   pcg_state/pcg_inc the generator's 128-bit state and increment as {high, low} 64-bit words
 *   proposals [n_chains][n_par], u [n_chains], n_draws = doubles consumed (advance the generator
 *   by this), n_failed [n_chains] failed attempts, fail_masks [n_chains][TRPL_MAX_LOGGED_FAILS]
 *   checks failed by each of the first failed attempts: bit i = parameter i out of bounds,
 *   bit 30 = p0 <= n0, bit 31 = tauN and tauP more than two decades apart.  n_par <= 30.
 *   idx_mun >= 0 switches on do_mu_constraint (trial_move_generation.py:77-83): every attempt takes
 *   the next of the caller's pre-drawn np.random uniforms ambi_u[n_ambi_u] (the reference draws the
 *   ambipolar mobility from the GLOBAL np.random stream), new_ambi = ambi_lo + (ambi_hi - ambi_lo) u,
 *   and mu_p is set from new_ambi and the proposed mu_n; n_ambi_used tells the caller how many to
 *   consume from np.random.  mu_arg [n_chains] receives the linear mu_p of each chain's final attempt:
 *   the caller overwrites proposals[:, idx_mup] with ITS log10 of it (NumPy's log10 is not libm's). */
#define TRPL_MAX_LOGGED_FAILS 8
int trpl_make_trial_moves(int32_t n_chains, int32_t n_par, const double* cur, const double* moves,
                          const uint8_t* do_log, const uint8_t* active, const double* lo,
                          const double* hi, int32_t idx_p0, int32_t idx_n0, int32_t idx_taun,
                          int32_t idx_taup, int32_t hard_bounds, int32_t max_tries,
                          const uint64_t pcg_state[2], const uint64_t pcg_inc[2], double* proposals,
                          double* u, int64_t* n_draws, int32_t* n_failed, uint32_t* fail_masks,
                          int32_t idx_mun, int32_t idx_mup, double ambi_lo, double ambi_hi,
                          const double* ambi_u, int32_t n_ambi_u, int32_t* n_ambi_used, double* mu_arg);

#ifdef __cplusplus
}
#endif
#endif /* METROTRPL_B200_H */
