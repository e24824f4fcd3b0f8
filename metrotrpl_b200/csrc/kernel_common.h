// kernel_common.h - what the translation units of the library share on the device side: the launch
// plan, the work queue, the trajectory tail and the tensor-memory slice of a warp.  The launch
// arguments and the per-trajectory glue the host lock-step build runs as well are in traj_io.h.
//   trpl_kernels.cu   one warp per trajectory (simt.h with TRPL_TEAM == 1), the C ABI
//   team_kernels.cu   a team of two warps per trajectory (TRPL_TEAM == 2): the grids of 129..256 nodes
//   team4_kernels.cu  a team of four warps per trajectory (TRPL_TEAM == 4): the grids of 257..512 nodes
// Included inside each unit after trajectory.h; everything here except LaunchPlan has internal linkage.
#pragma once
#include <cuda_runtime.h>
#include "traj_io.h"

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

// step-log / scratch slot of the warp, team or CTA `i` of this CTA
__device__ __forceinline__ unsigned cta_slot(const KernelArgs& a, int i) { return blockIdx.x * a.slots_per_cta + i; }

// tail-only addresses are formed after the loop from the (constant-bank) launch arguments
__device__ __forceinline__ void finish_traj(const KernelArgs& a, int traj, unsigned slot, const TrajIn& in,
                                            const TrajMid& mid, TrajOut& out) {
  TailIn tl;
  tail_in(a, in, traj, slot, tl);
  finalize_trajectory(in, tl, a.opt, mid, out);
  if ((threadIdx.x & (unsigned)(simt::LANES - 1)) == 0) store_result(a, traj, out);
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
