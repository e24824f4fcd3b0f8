// trpl_emu_fit.cpp - host lock-step build of the fitted-curve pass (TRPL_OPT_FIT): the routine the
// library's trpl_fit_kernel runs on the stored curves (trajectory.h fit_trajectory), compiled with
// TRPL_HOST_EMU on the one-warp vocabulary, as that kernel is.  Test infrastructure only, built and
// loaded by tests/emu/fit_emu.py.  Takes the curves of a run of the host build (trpl_emu.cpp).
#define TRPL_HOST_EMU 1
#include <stdint.h>
#include <string.h>
#include <cmath>
#include <vector>
#include "../../include/metrotrpl_b200.h"
#include "../../metrotrpl_b200/csrc/trajectory.h"

using namespace trpl;

extern "C" int trpl_emu_fit_batch(int32_t n_meas, const trpl_meas_desc* meas, int32_t n_times_total,
                                  const double* times, const double* vals, const double* uncs, int32_t n_sets,
                                  const double* aux, const trpl_solver_opts* opts, const double* curves,
                                  const double* irf_mom, double* fit) {
  static_assert(sizeof(trpl_meas_desc) == sizeof(MeasDesc), "ABI struct mismatch");
  if (!vals || !uncs || !curves || !fit) return 1;
  SolverOpts opt;
  memcpy(&opt, opts, sizeof(opt));
  const MeasDesc* mds = reinterpret_cast<const MeasDesc*>(meas);
  const int n_traj = n_sets * n_meas;
#pragma omp parallel for schedule(dynamic, 1)
  for (int traj = 0; traj < n_traj; ++traj) {
    const int set = traj / n_meas, mi = traj % n_meas;
    const MeasDesc* md = mds + mi;
    // the fields fit_trajectory reads, set as the library's setup_traj sets them
    TrajIn in;
    memset(&in, 0, sizeof(in));
    in.md = md;
    in.times = times + md->t_off;
    in.vals = vals + md->t_off;
    in.uncs = uncs + md->t_off;
    const double* ax = aux + (size_t)traj * TRPL_NAUX;
    in.scale_shift = ax[TRPL_A_SCALE_SHIFT];
    in.s2T[0] = ax[TRPL_A_S2T0]; in.s2T[1] = ax[TRPL_A_S2T1]; in.s2T[2] = ax[TRPL_A_S2T2];
    in.curve = const_cast<double*>(curves) + (size_t)set * n_times_total + md->t_off;
    TailIn tl;
    memset(&tl, 0, sizeof(tl));
    std::vector<double> ry, hk, trim;
    tl.irf.nk = (irf_mom && md->irf_nk > 0) ? md->irf_nk : 0;
    tl.irf.dt = md->irf_dt;
    tl.irf.mom = irf_mom ? irf_mom + 3 * (size_t)md->irf_off : nullptr;
    if (tl.irf.nk > 0) {
      const double tend = in.times[md->n_t - 1];
      const size_t n_rs = (size_t)ceil((tend + md->irf_dt / 4) / (md->irf_dt / 2));
      ry.resize(n_rs + 4); hk.resize(n_rs / 2 + 4); trim.resize(md->n_t + 4);
    }
    tl.irf.ry = ry.data(); tl.irf.hk = hk.data(); tl.irf.trim = trim.data();
    fit_trajectory(in, tl, opt, fit + (size_t)set * n_times_total + md->t_off);
  }
  return 0;
}
