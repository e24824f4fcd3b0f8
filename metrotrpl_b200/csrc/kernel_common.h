// kernel_common.h - what the translation units of the library share: the launch arguments and plan,
// the work queue, the per-trajectory set-up / result write-back and the tensor-memory slice of a warp.
//   trpl_kernels.cu   one warp per trajectory (simt.h with TRPL_TEAM == 1), the C ABI
//   team_kernels.cu   a team of two warps per trajectory (TRPL_TEAM == 2): the grids of 129..256 nodes
//   team4_kernels.cu  a team of four warps per trajectory (TRPL_TEAM == 4): the grids of 257..512 nodes
// Included inside each unit after trajectory.h; everything here except LaunchPlan has internal linkage.
#pragma once
#include <cuda_runtime.h>
#include "../../include/metrotrpl_b200.h"
#include "trajectory.h"

// How one launch of a persistent trajectory kernel is shaped (run_plan in trpl_kernels.cu runs it).
// Global scope: the team units fill it for their kernels, so every unit sees one layout.
struct LaunchPlan {
  const void* kernel;            // first pass
  const void* explicit_kernel;   // second pass over the trajectories the first deferred, or null
  int block;                     // threads per CTA
  size_t smem;                   // dynamic shared memory per CTA (0: static only)
  int tm_cols;                   // tensor-memory columns per CTA (0: none)
  int traj_per_cta;              // concurrent trajectories per CTA = step-log / scratch slices per CTA
};

namespace {

using namespace trpl;

// Residency: 8 trajectories per SM - two CTAs of four warps at 255 registers per thread.  (Twelve
// per SM at 168 registers, with the tensor-memory slices of a 12-warp CTA stacked along the
// columns, was built and measured: no gain, DESIGN.md section 5.)
constexpr int WARPS_PER_CTA = 4;                  // one warp per tensor-memory lane quarter
constexpr int CTAS_PER_SM = 2;
constexpr int pow2_cols(int c) { return c == 0 ? 0 : c <= 32 ? 32 : c <= 64 ? 64 : c <= 128 ? 128 : c <= 256 ? 256 : 512; }

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

// Queue position -> trajectory index (results are indexed [set][meas]).  Without an explicit order
// the queue is measurement-major with the (statically) most expensive curves first, so that the
// tail of the launch is made of the cheapest trajectories.
__device__ __forceinline__ int queue_traj(const KernelArgs& a, int q) {
  if (a.queue) return a.queue[q];
  const int n_sets_q = a.n_traj / a.n_meas;
  const int qm = q / n_sets_q;
  return (q - qm * n_sets_q) * a.n_meas + a.meas_order[qm];
}

// next queue position of a warp: lane 0 claims it, every lane receives it
__device__ __forceinline__ int warp_claim(int* counter, int lane) {
  int q = 0;
  if (lane == 0) q = atomicAdd(counter, 1);
  return __shfl_sync(0xffffffffu, q, 0);
}

// next queue position of a CTA: thread 0 claims it into the __shared__ `slot`, every thread reads it
__device__ __forceinline__ int cta_claim(int* counter, int* slot) {
  __syncthreads();
  if (threadIdx.x == 0) *slot = atomicAdd(counter, 1);
  __syncthreads();
  return *slot;
}

__device__ __forceinline__ void setup_traj(const KernelArgs& a, int traj, int warp, TrajIn& in) {
  in.hist = a.hist + (size_t)(blockIdx.x * a.slots_per_cta + warp) * (3 * HIST_CAP);
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

// tail-only addresses are formed after the loop from the (constant-bank) launch arguments
__device__ __forceinline__ void finish_traj(const KernelArgs& a, int traj, int warp, const TrajIn& in,
                                            const TrajMid& mid, TrajOut& out) {
  const MeasDesc* md = in.md;
  const bool conv = a.irf_mom && a.scratch && md->irf_nk > 0;
  const bool ladder = (a.opt.flags & OPT_LADDER) && a.n_ladder > 0 && a.scratch;
  TailIn tl;
  tl.irf.nk = conv ? md->irf_nk : 0;
  tl.irf.dt = md->irf_dt;
  tl.irf.mom = a.irf_mom ? a.irf_mom + 3 * (size_t)md->irf_off : nullptr;
  double* ws = a.scratch ? a.scratch + (size_t)(blockIdx.x * a.slots_per_cta + warp) * a.scratch_stride : nullptr;
  tl.irf.ry = ws; tl.irf.hk = ws ? ws + a.off_hk : nullptr; tl.irf.trim = ws ? ws + a.off_trim : nullptr;
  tl.r2_scratch = (ws && ladder) ? ws + a.off_r2 : nullptr;
  tl.u2_scratch = (ws && ladder) ? ws + a.off_u2 : nullptr;
  tl.ladder_T = a.ladder_T; tl.ladder_n = a.n_ladder;
  tl.ladder_out = a.ladder_out ? a.ladder_out + (size_t)traj * a.n_ladder : nullptr;
  finalize_trajectory(in, tl, a.opt, mid, out);
  if ((threadIdx.x & (unsigned)(simt::LANES - 1)) == 0) {
    a.logll[3 * (size_t)traj + 0] = out.logll[0];
    a.logll[3 * (size_t)traj + 1] = out.logll[1];
    a.logll[3 * (size_t)traj + 2] = out.logll[2];
    a.status[traj] = out.status;
    a.nsteps[2 * (size_t)traj + 0] = out.n_acc;
    a.nsteps[2 * (size_t)traj + 1] = out.n_rej;
  }
  warp_sync();
}

// Tensor-memory slice of the calling warp.  One warp of the CTA allocates TM_COLS columns for the
// CTA (tcgen05.alloc hands out whole columns, all 128 lanes); warp w then owns lanes 32*(w%4)..+31
// of those columns.  A CTA has at most four warps, so the slices are disjoint.
template <class SL>
struct TmCta {
  static constexpr int COLS = pow2_cols(4 * SL::TM_COUNT);   // columns one CTA allocates
  static_assert(4 * SL::TM_COUNT <= 512, "tensor-memory slice exceeds 512 columns");
};
template <class SL>
__device__ __forceinline__ LaneTm tmem_acquire(int warp) {
  LaneTm tm{0u};
  if constexpr (SL::TM_COUNT > 0) {
    __shared__ unsigned tm_base_s;
    if (warp == 0) {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                   :: "r"((unsigned)__cvta_generic_to_shared(&tm_base_s)), "n"(TmCta<SL>::COLS) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    // broadcast from lane 0: tells ptxas the address is warp-uniform (it then lives in a uniform
    // register instead of being re-derived from the thread index in front of every access)
    tm.base = __shfl_sync(0xffffffffu, tm_base_s + ((unsigned)(32 * warp) << 16), 0);
  }
  return tm;
}
// every warp of the CTA is done with its slice: the allocating warp gives the columns back
template <class SL>
__device__ __forceinline__ void tmem_release(int warp, const LaneTm& tm) {
  if constexpr (SL::TM_COUNT > 0) {
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0)      // warp 0 owns lane quarter 0: its base is the allocation
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;"
                   :: "r"(tm.base), "n"(TmCta<SL>::COLS) : "memory");
  }
}


}  // namespace
