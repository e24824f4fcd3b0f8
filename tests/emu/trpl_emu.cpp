// trpl_emu.cpp - host lock-step build of the SAME integrator source the CUDA kernel compiles
// (metrotrpl_b200/csrc/trajectory.h) with TRPL_HOST_EMU.  Test infrastructure only: it lets the
// CPU-only test tier exercise the warp algorithm (partition + PCR solve, RODAS4 controller, Hermite
// readout, likelihood) against the oracle.  A run is planned, set up and written back by the
// library's own code (traj_io.h): the same stored outputs, the same per-slot scratch layout, one slot
// per OpenMP thread.  It is built and loaded by tests/ only and is never reachable from the
// metrotrpl_b200 package.
#define TRPL_HOST_EMU 1
#include <omp.h>
#include <stdint.h>
#include <string.h>
#include <algorithm>
#include <vector>
#include "../../metrotrpl_b200/csrc/traj_io.h"
#include "../../metrotrpl_b200/csrc/explicit.h"
#if TRPL_TEAM == 1
#include "../../metrotrpl_b200/csrc/extrapolation.h"
#endif

template <int NPL, int MODEL, bool FULL>
static void run_all(const KernelArgs& a) {
#pragma omp parallel
  {
    const unsigned slot = omp_get_thread_num();
#pragma omp for schedule(dynamic, 1)
    for (int traj = 0; traj < a.n_traj; ++traj) {
      TrajMem sm{simt::LaneMem(Slots<NPL, MODEL>::COUNT), simt::LaneTm(Slots<NPL, MODEL>::TM_COUNT)};
      TrajIn in;
      setup_traj(a, traj, slot, in);
      TrajOut out;
      TrajMid mid;
#if TRPL_TEAM == 1
      if (a.opt.flags & OPT_EXTRAPOLATION) {
        run_trajectory_seulex<NPL, MODEL, FULL>(in, a.opt, sm, out, mid);      // the one-warp driver
      } else
#endif
      if (run_trajectory<NPL, MODEL, FULL>(in, a.opt, sm, out, mid, !(a.opt.flags & OPT_NO_EXPLICIT))) {
        run_trajectory_explicit<NPL, MODEL, FULL>(in, a.opt, sm, out, mid);
        out.status |= ST_EXPLICIT;
      }
      TailIn tl;
      tail_in(a, in, traj, slot, tl);
      finalize_trajectory(in, tl, a.opt, mid, out);
      store_result(a, traj, out);
    }
    // the fit pass reads the curves of every trajectory: after the loop's closing barrier
    if (a.fit) {
#pragma omp for schedule(dynamic, 1)
      for (int traj = 0; traj < a.n_traj; ++traj) {
        TrajIn in;
        setup_traj(a, traj, slot, in);
        TailIn tl;
        tail_in(a, in, traj, slot, tl);
        fit_trajectory(in, tl, a.opt, a.fit + (size_t)(traj / a.n_meas) * a.n_times_total + in.md->t_off);
      }
    }
  }
}

template <int MODEL>
static const char* dispatch(int max_nx, bool all_full, const KernelArgs& a) {
#define GO(N, F) run_all<N, MODEL, F>(a)
#if TRPL_TEAM >= 2
  // the team vocabularies (team_kernels.cu / team4_kernels.cu): 64 or 128 lanes x 4 nodes, the grids
  // of 129..256 / 257..512 nodes
  constexpr int TOP = 128 * TRPL_TEAM;
  if (all_full && max_nx == TOP) GO(4, true);
  else if (max_nx > TOP / 2 && max_nx <= TOP) GO(4, false);
  else return "nx outside the grids of this team build";
#else
  // (8 nodes per lane: no product kernel any more, kept for the generic one-warp extrapolation driver)
  if (all_full && max_nx == 128) GO(4, true);
  else if (all_full && max_nx == 256) GO(8, true);
  else if (max_nx <= 32) GO(1, false);
  else if (max_nx <= 64) GO(2, false);
  else if (max_nx <= 128) GO(4, false);
  else if (max_nx <= 256) GO(8, false);
  else return "nx > 256 needs a team build";
#endif
#undef GO
  return nullptr;
}

// The library's trpl_set_problem + trpl_set_irf + trpl_set_ladder + trpl_loglik_batch on host arrays:
// curves, ladder_out and fit are the outputs of the run (null: not wanted).  Returns null, or the
// message the run is refused with.
extern "C" const char* trpl_emu_loglik_batch(int32_t model, int32_t n_meas, const trpl_meas_desc* meas,
                                             int32_t n_times_total, const double* times, const double* vals,
                                             const double* uncs, const double* profiles, int32_t n_sets,
                                             const double* params, const double* aux,
                                             const trpl_solver_opts* opts, double* logll, int32_t* status,
                                             int32_t* nsteps, double* curves, const double* irf_mom,
                                             const double* ladder_T, int32_t n_ladder, double* ladder_out,
                                             double* fit) {
  static_assert(sizeof(trpl_meas_desc) == sizeof(MeasDesc), "ABI struct mismatch");
  const MeasDesc* md = reinterpret_cast<const MeasDesc*>(meas);
  ProblemFacts pf{vals && uncs, false, irf_mom != nullptr, ladder_T ? n_ladder : 0, 0, 0};
  int max_nx = 0;
  for (int i = 0; i < n_meas; ++i) {
    if (md[i].nx < 2 || md[i].nx > 512) return "nx must be in 2..512";
    max_nx = std::max(max_nx, md[i].nx);
    pf.max_nt = std::max(pf.max_nt, (size_t)md[i].n_t);
    if (md[i].irf_nk > 0) {
      pf.any_irf = true;
      pf.max_nrs = std::max(pf.max_nrs, (size_t)irf_resample_count(times[md[i].t_off + md[i].n_t - 1], md[i].irf_dt));
    }
  }
  // trpl_set_problem's rule: rhs and jacobian (model.h) need the two contacts on different lanes
  const int npl = max_nx <= 32 ? 1 : max_nx <= 64 ? 2 : 4;
  for (int i = 0; i < n_meas; ++i)
    if (md[i].nx <= npl) return "mixed nx: smallest nx must exceed the nodes per lane of the largest grid (1, 2 or 4)";
  bool all_full = true;
  for (int i = 0; i < n_meas; ++i) if (md[i].nx != max_nx) all_full = false;
  RunPlan p;
  if (const char* why = plan_run(pf, opts->flags, curves != nullptr, p)) return why;
  if ((p.ladder && !ladder_out) || (p.fit && !fit)) return "no output array for the ladder rows or the fit";
  std::vector<double> own_curves(p.curves && !curves ? (size_t)n_sets * n_times_total : 0);
  const int n_slots = omp_get_max_threads();
  std::vector<double> scratch(n_slots * p.scratch_stride), hist((size_t)n_slots * 3 * HIST_CAP);
  KernelArgs a{};
  a.params = params; a.aux = aux; a.meas = md; a.times = times;
  a.vals = pf.have_vals ? vals : nullptr; a.uncs = pf.have_vals ? uncs : nullptr;
  a.profiles = profiles;
  a.logll = logll; a.status = status; a.nsteps = nsteps;
  p.set_args(a, curves ? curves : own_curves.data(), irf_mom, ladder_T, ladder_out, n_ladder, fit);
  if (p.scratch_stride > 0) a.scratch = scratch.data();
  a.hist = hist.data();
  a.n_traj = n_sets * n_meas; a.n_meas = n_meas; a.n_times_total = n_times_total;
  memcpy(&a.opt, opts, sizeof(SolverOpts));
  if (model == TRPL_MODEL_STD) return dispatch<MODEL_STD>(max_nx, all_full, a);
  return dispatch<MODEL_TRAPS>(max_nx, all_full, a);
}
