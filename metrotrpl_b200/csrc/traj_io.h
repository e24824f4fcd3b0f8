// traj_io.h - the per-run and per-trajectory glue of the trajectory kernels that needs neither the
// CUDA runtime nor tensor memory: the launch arguments, what a run stores and how its scratch is laid
// out, a trajectory's inputs and tail set-up from its index, and its result write-back.  The library's
// kernels (kernel_common.h) and the host lock-step build (tests/emu/trpl_emu.cpp) both run these, so
// the host build makes the same decisions on the same layout.
// Included after trajectory.h; everything here has internal linkage.
#pragma once
#include "../../include/metrotrpl_b200.h"
#include "trajectory.h"

namespace {

using namespace trpl;

struct KernelArgs {
  const double* params;      // [n_sets][16]
  const double* aux;         // [n_sets][n_meas][6]
  const MeasDesc* meas;      // [n_meas]
  const double* times;
  const double* vals;
  const double* uncs;
  const double* profiles;
  double* logll;             // [n_traj][3]
  int* status;               // [n_traj]
  int* nsteps;               // [n_traj][2]
  double* curves;            // [n_sets][n_times_total] or null
  const double* irf_mom;     // [rows][3] or null
  double* scratch;           // per-slot slices: resampled | convolved | trimmed
  size_t scratch_stride, off_hk, off_trim, off_r2, off_u2;
  const double* ladder_T;
  double* ladder_out;        // [n_traj][n_ladder]
  int n_ladder;
  int* counter;              // work queue head
  const int* meas_order;     // [n_meas] measurement indices, most expensive first
  const int* queue;          // [n_traj] explicit queue order (trpl_set_queue_order) or null
  double* hist;              // per-slot step histories, 3 * HIST_CAP doubles each
  int* defer_list;           // trajectories handed to the explicit path
  int* defer_count;
  int n_traj, n_meas, n_times_total;
  int slots_per_cta;         // trajectories a CTA runs at once (warps, teams or 1): step-log / scratch slices
  SolverOpts opt;
  double* fit;               // [n_sets][n_times_total] fitted curves (TRPL_OPT_FIT, trpl_fit_kernel) or null
};

// What trpl_set_problem, trpl_set_irf and trpl_set_ladder record that a run's plan depends on.
struct ProblemFacts {
  bool have_vals, any_irf, have_irf;
  int n_ladder;
  size_t max_nrs, max_nt;    // longest resampled IRF curve, most measurement times
};

// What one run stores besides the results, and the layout of its per-slot scratch.
struct RunPlan {
  bool curves, conv, ladder, fit;
  size_t scratch_stride, off_hk, off_trim, off_r2, off_u2;    // stride 0: no scratch

  // the plan's part of the launch arguments: the buffers the run does not use stay null (a.scratch
  // too: the caller points it at the slices once it knows how many there are)
  void set_args(KernelArgs& a, double* curves_buf, const double* irf_mom, const double* ladder_T,
                double* ladder_out, int n_ladder, double* fit_buf) const {
    a.curves = curves ? curves_buf : nullptr;
    a.irf_mom = conv ? irf_mom : nullptr;
    a.scratch = nullptr;
    a.scratch_stride = scratch_stride; a.off_hk = off_hk; a.off_trim = off_trim; a.off_r2 = off_r2; a.off_u2 = off_u2;
    a.ladder_T = ladder ? ladder_T : nullptr;
    a.ladder_out = ladder ? ladder_out : nullptr;
    a.n_ladder = ladder ? n_ladder : 0;
    a.fit = fit ? fit_buf : nullptr;
  }
};

// Plans a run with option flags `flags`.  Returns null, or the message the run is refused with.
inline const char* plan_run(const ProblemFacts& pf, int flags, bool want_curves, RunPlan& p) {
  const bool want_ll = !(flags & OPT_NO_LIKELIHOOD);
  p = RunPlan{};
  p.fit = (flags & OPT_FIT) != 0;
  if (p.fit && !want_ll)
    return "TRPL_OPT_FIT returns what the likelihood compares: it cannot be combined with TRPL_OPT_NO_LIKELIHOOD";
  if (p.fit && !pf.have_vals) return "TRPL_OPT_FIT needs measurement values (vals, uncs in trpl_set_problem)";
  if (want_ll && !pf.have_vals) return "likelihood requested but no measurement values uploaded";
  p.conv = want_ll && pf.any_irf;
  if (p.conv && !pf.have_irf) return "measurements ask for IRF convolution but trpl_set_irf was not called";
  p.ladder = want_ll && (flags & OPT_LADDER);
  if (p.ladder && pf.n_ladder < 1) return "TRPL_OPT_LADDER without trpl_set_ladder";
  // the min_y pass, the convolution, the ladder and the fit pass re-read the stored curve
  p.curves = want_curves || (flags & OPT_FORCE_MIN_Y) || p.conv || p.ladder || p.fit;
  if (p.conv || p.ladder) {
    // per-slot scratch: resampled | convolved | trimmed curve | residuals^2 | 2 unc^2 (all stay in L2)
    const size_t nrs = p.conv ? pf.max_nrs : 0;
    const size_t n_hk = p.conv ? (pf.max_nrs - 1) / 2 + 1 : 0;
    const size_t nt4 = (pf.max_nt + 3) & ~(size_t)3;
    p.off_hk = (nrs + 3) & ~(size_t)3;
    p.off_trim = p.off_hk + ((n_hk + 3) & ~(size_t)3);
    p.off_r2 = p.off_trim + nt4;
    p.off_u2 = p.off_r2 + nt4;
    p.scratch_stride = p.off_u2 + nt4;
  }
  return nullptr;
}

// Inputs of trajectory `traj` ([set][meas]); `slot` is its step-log / scratch slice (unsigned: on the
// device it is formed from blockIdx.x).
TRPL_FN void setup_traj(const KernelArgs& a, int traj, unsigned slot, TrajIn& in) {
  in.hist = a.hist + (size_t)slot * (3 * HIST_CAP);
  const int set = traj / a.n_meas;
  const int mi = traj - set * a.n_meas;
  const MeasDesc* md = a.meas + mi;
  in.par = a.params + (size_t)set * TRPL_NPARAM;
  in.md = md;
  in.times = a.times + md->t_off;
  in.vals = a.vals ? a.vals + md->t_off : nullptr;
  in.uncs = a.uncs ? a.uncs + md->t_off : nullptr;
  in.profile = a.profiles ? a.profiles + md->prof_off : nullptr;
  const double* ax = a.aux + (size_t)traj * TRPL_NAUX;
  in.scale_shift = ax[TRPL_A_SCALE_SHIFT];
  in.s2T[0] = ax[TRPL_A_S2T0]; in.s2T[1] = ax[TRPL_A_S2T1]; in.s2T[2] = ax[TRPL_A_S2T2];
  in.fl_mult = ax[TRPL_A_FLUENCE_MULT]; in.al_mult = ax[TRPL_A_ABSORB_MULT];
  in.curve = a.curves ? a.curves + (size_t)set * a.n_times_total + md->t_off : nullptr;
  const bool want_ll = !(a.opt.flags & OPT_NO_LIKELIHOOD);
  const bool conv = a.irf_mom && a.scratch && md->irf_nk > 0;
  const bool ladder = (a.opt.flags & OPT_LADDER) && a.n_ladder > 0 && a.scratch;
  in.post_pass = want_ll && in.curve && ((a.opt.flags & OPT_FORCE_MIN_Y) || conv || ladder);
}

// What only the final pass of the trajectory `in` was set up for needs: its IRF and ladder scratch
// in slice `slot`, its ladder row.
TRPL_FN void tail_in(const KernelArgs& a, const TrajIn& in, int traj, unsigned slot, TailIn& tl) {
  const MeasDesc* md = in.md;
  const bool conv = a.irf_mom && a.scratch && md->irf_nk > 0;
  const bool ladder = (a.opt.flags & OPT_LADDER) && a.n_ladder > 0 && a.scratch;
  tl.irf.nk = conv ? md->irf_nk : 0;
  tl.irf.dt = md->irf_dt;
  tl.irf.mom = a.irf_mom ? a.irf_mom + 3 * (size_t)md->irf_off : nullptr;
  double* ws = a.scratch ? a.scratch + (size_t)slot * a.scratch_stride : nullptr;
  tl.irf.ry = ws; tl.irf.hk = ws ? ws + a.off_hk : nullptr; tl.irf.trim = ws ? ws + a.off_trim : nullptr;
  tl.r2_scratch = (ws && ladder) ? ws + a.off_r2 : nullptr;
  tl.u2_scratch = (ws && ladder) ? ws + a.off_u2 : nullptr;
  tl.ladder_T = a.ladder_T; tl.ladder_n = a.n_ladder;
  tl.ladder_out = a.ladder_out ? a.ladder_out + (size_t)traj * a.n_ladder : nullptr;
}

TRPL_FN void store_result(const KernelArgs& a, int traj, const TrajOut& out) {
  a.logll[3 * (size_t)traj + 0] = out.logll[0];
  a.logll[3 * (size_t)traj + 1] = out.logll[1];
  a.logll[3 * (size_t)traj + 2] = out.logll[2];
  a.status[traj] = out.status;
  a.nsteps[2 * (size_t)traj + 0] = out.n_acc;
  a.nsteps[2 * (size_t)traj + 1] = out.n_rej;
}

}  // namespace
