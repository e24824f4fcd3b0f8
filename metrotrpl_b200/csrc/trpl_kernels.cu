// trpl_kernels.cu - sm_100a kernels and the C ABI (include/metrotrpl_b200.h).
//
// Execution model: persistent warps.  The grid is (SM count x 2) CTAs of 4 warps; every warp
// repeatedly claims the next (parameter set, measurement) trajectory from a global counter and
// integrates it start to finish (trajectory.h) using only its registers, its private slice of
// tensor memory (factor blocks, PCR multipliers: lane-private data) and its private slice of shared
// memory (stage increments, lane exchange).  The only __syncthreads are the two that bracket the
// CTA's tensor-memory allocation, there is no inter-warp communication, and the only global
// traffic per trajectory is its 16 parameters, the measurement arrays (L2-resident, shared by all
// trajectories), its step log and a handful of result scalars.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <string>
#include <vector>
#include <algorithm>
#include <cmath>

#include "../../include/metrotrpl_b200.h"
#include "trajectory.h"
#include "explicit.h"
#include "cta_trajectory.h"
#include "extrapolation.h"
#include "proposals.h"

#include "kernel_common.h"

namespace {

static_assert(sizeof(trpl_meas_desc) == sizeof(MeasDesc), "ABI struct mismatch");
static_assert(sizeof(trpl_solver_opts) == sizeof(SolverOpts), "ABI struct mismatch");
static_assert(TRPL_NPARAM == trpl::NPARAM, "ABI constant mismatch");

template <int NPL, int MODEL, bool FULL>
__global__ void __launch_bounds__(32 * WARPS_PER_CTA, CTAS_PER_SM) trpl_forward_kernel(const KernelArgs a) {
  typedef Slots<NPL, MODEL> SL;
  extern __shared__ double2 smem[];
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);     // warp-uniform by construction
  const int lane = threadIdx.x & 31;
  TrajMem mem{LaneMem{smem + warp * (SL::COUNT * 32)}, tmem_acquire<SL>(warp)};   // COUNT pairs of 16 B per lane
  const bool allow_defer = a.defer_list != nullptr;
  for (;;) {
    const int q = warp_claim(a.counter, lane);
    if (q >= a.n_traj) break;
    const int traj = queue_traj(a, q);
    TrajIn in;
    setup_traj(a, traj, cta_slot(a, warp), in);
    TrajOut out;
    TrajMid mid;
    if (run_trajectory<NPL, MODEL, FULL>(in, a.opt, mem, out, mid, allow_defer)) {
      if (lane == 0) a.defer_list[atomicAdd(a.defer_count, 1)] = traj;     // non-stiff: explicit path
      continue;
    }
    finish_traj(a, traj, cta_slot(a, warp), in, mid, out);
  }
  tmem_release<SL>(warp, mem.tm);
}

// second pass over the trajectories the first kernel classified non-stiff
template <int NPL, int MODEL, bool FULL>
__global__ void __launch_bounds__(32 * WARPS_PER_CTA, CTAS_PER_SM) trpl_explicit_kernel(const KernelArgs a) {
  typedef Slots<NPL, MODEL> SL;
  extern __shared__ double2 smem[];
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;
  TrajMem mem{LaneMem{smem + warp * (SL::COUNT * 32)}, tmem_acquire<SL>(warp)};
  const int n = *a.defer_count;
  for (;;) {
    const int q = warp_claim(a.counter + 1, lane);
    if (q >= n) break;
    const int traj = a.defer_list[q];
    TrajIn in;
    setup_traj(a, traj, cta_slot(a, warp), in);
    TrajOut out;
    TrajMid mid;
    run_trajectory_explicit<NPL, MODEL, FULL>(in, a.opt, mem, out, mid);
    out.status |= ST_EXPLICIT;
    finish_traj(a, traj, cta_slot(a, warp), in, mid, out);
  }
  tmem_release<SL>(warp, mem.tm);
}

// The order-6 extrapolation integrator (extrapolation.h), one warp per trajectory: persistent warps
// exactly like trpl_forward_kernel (same storage layout, same queue).  Exists for A/B measurements
// and as the bit-for-bit twin of the cooperative kernel below.
template <int NPL, int MODEL, bool FULL>
__global__ void __launch_bounds__(32 * WARPS_PER_CTA, CTAS_PER_SM) trpl_seulex_kernel(const KernelArgs a) {
  typedef Slots<NPL, MODEL> SL;
  extern __shared__ double2 smem[];
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;
  TrajMem mem{LaneMem{smem + warp * (SL::COUNT * 32)}, tmem_acquire<SL>(warp)};
  for (;;) {
    const int q = warp_claim(a.counter, lane);
    if (q >= a.n_traj) break;
    const int traj = queue_traj(a, q);
    TrajIn in;
    setup_traj(a, traj, cta_slot(a, warp), in);
    TrajOut out;
    TrajMid mid;
    run_trajectory_seulex<NPL, MODEL, FULL>(in, a.opt, mem, out, mid);
    finish_traj(a, traj, cta_slot(a, warp), in, mid, out);
  }
  tmem_release<SL>(warp, mem.tm);
}

// The same integrator with the six columns of every step spread over the four warps of the CTA:
// ONE trajectory per CTA, a quarter of the sequential depth.  Each warp keeps the full state and its
// own factorisation storage (its slices of tensor and shared memory, as in trpl_forward_kernel); the
// increments of the columns cross warps through an exchange area behind the slices (SeulexXch:
// double-buffered for 'std', single-buffered for traps).
template <int NPL, int MODEL, bool FULL>
__global__ void __launch_bounds__(32 * WARPS_PER_CTA, CTAS_PER_SM) trpl_seulex_cta_kernel(const KernelArgs a) {
  typedef Slots<NPL, MODEL> SL;
  extern __shared__ double2 smem[];
  __shared__ int s_traj, s_flag;
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  TrajMem mem{LaneMem{smem + warp * (SL::COUNT * 32)}, tmem_acquire<SL>(warp)};
  double2* xch = smem + WARPS_PER_CTA * (SL::COUNT * 32);
  for (;;) {
    const int q = cta_claim(a.counter, &s_traj);
    if (q >= a.n_traj) break;
    const int traj = queue_traj(a, q);
    TrajIn in;
    setup_traj(a, traj, cta_slot(a, 0), in);    // slots_per_cta == 1: one step log / scratch slice per CTA
    TrajOut out;
    TrajMid mid;
    run_trajectory_seulex_cta<NPL, MODEL, FULL>(in, a.opt, mem, xch, &s_flag, warp, out, mid);
    if (warp == 0) finish_traj(a, traj, cta_slot(a, 0), in, mid, out);
  }
  tmem_release<SL>(warp, mem.tm);
}

// One trajectory per CTA of 128 threads (cta_trajectory.h): the low-latency instantiation for small
// batches.  Persistent CTAs claim trajectories from the same queue as the one-warp kernel.
__global__ void __launch_bounds__(cta::NX, 2) trpl_cta_kernel(const KernelArgs a) {
  __shared__ cta::Smem s;
  for (;;) {
    const int q = cta_claim(a.counter, &s.traj);
    if (q >= a.n_traj) break;
    const int traj = queue_traj(a, q);
    TrajIn in;
    setup_traj(a, traj, cta_slot(a, 0), in);
    TrajOut out;
    TrajMid mid;
    cta::run_trajectory_cta(in, a.opt, s, out, mid);
    if (threadIdx.x < 32) finish_traj(a, traj, cta_slot(a, 0), in, mid, out);
  }
}

// TRPL_OPT_FIT: the fitted curve of every trajectory (trajectory.h fit_trajectory), from the curves
// the trajectory kernel stored.  Runs after it on the same stream, one warp per CTA, each CTA in its
// own scratch slice (launched with at most as many CTAs as the trajectory kernel had slices).  The
// convolution is set up as in tail_in, with the CTA's slice formed once, before the loop.
__global__ void __launch_bounds__(32) trpl_fit_kernel(const KernelArgs a) {
  double* ws = a.scratch ? a.scratch + (size_t)blockIdx.x * a.scratch_stride : nullptr;
  for (int traj = blockIdx.x; traj < a.n_traj; traj += gridDim.x) {
    TrajIn in;
    setup_traj(a, traj, blockIdx.x, in);
    const MeasDesc* md = in.md;
    TailIn tl;
    tl.irf.nk = (a.irf_mom && ws && md->irf_nk > 0) ? md->irf_nk : 0;
    tl.irf.dt = md->irf_dt;
    tl.irf.mom = a.irf_mom ? a.irf_mom + 3 * (size_t)md->irf_off : nullptr;
    tl.irf.ry = ws; tl.irf.hk = ws ? ws + a.off_hk : nullptr; tl.irf.trim = ws ? ws + a.off_trim : nullptr;
    const int set = traj / a.n_meas;
    fit_trajectory(in, tl, a.opt, a.fit + (size_t)set * a.n_times_total + in.md->t_off);
  }
}

// Replica exchange needs each chain's likelihood at every ladder temperature summed over its
// measurements (the reference sums ll_func[ss](T) over ss, metropolis.py:73-76): [n_sets][n_temps].
// NaN (a failed curve) becomes -inf, as eval_trial_move's callers treat it.
__global__ void ladder_sum_kernel(const double* lad, double* out, int n_sets, int n_meas, int n_temps) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n_sets * n_temps) return;
  const int set = k / n_temps, tt = k - set * n_temps;
  double acc = 0.0;
  for (int m = 0; m < n_meas; ++m) acc += lad[((size_t)set * n_meas + m) * n_temps + tt];
  out[k] = (acc != acc) ? -HUGE_VAL : acc;
}

// FP64 peak probe: 8 independent FMA chains per thread, no memory traffic.
__global__ void __launch_bounds__(256) fp64_probe_kernel(double* out, int iters, double seed) {
  double a0 = seed, a1 = seed + 1, a2 = seed + 2, a3 = seed + 3, a4 = seed + 4, a5 = seed + 5,
         a6 = seed + 6, a7 = seed + 7;
  const double m = 0.999999, c = 1e-9 * threadIdx.x;
  for (int i = 0; i < iters; ++i) {
    a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
    a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
  }
  const double s = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
  if (s == 123.456) out[blockIdx.x * blockDim.x + threadIdx.x] = s;   // never true; defeats DCE
}

thread_local std::string g_err;
int fail(const std::string& msg) { g_err = msg; return 1; }
#define CU(call)                                                                             \
  do {                                                                                       \
    cudaError_t e_ = (call);                                                                 \
    if (e_ != cudaSuccess) return fail(std::string(#call) + ": " + cudaGetErrorString(e_)); \
  } while (0)

template <class T>
struct DevBuf {
  T* p = nullptr;
  size_t cap = 0;
  cudaError_t reserve(size_t n) {
    if (n <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr; cap = 0;
    cudaError_t e = cudaMalloc(&p, n * sizeof(T));
    if (e == cudaSuccess) cap = n;
    return e;
  }
  ~DevBuf() { if (p) cudaFree(p); }
};

}  // namespace

struct trpl_handle {
  int device = 0;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, tm0 = nullptr, tm1 = nullptr;
  DevBuf<char> d_flush;
  cudaDeviceProp prop;
  int model = 0, n_meas = 0, n_times_total = 0, max_nx = 0;
  bool have_vals = false, have_profiles = false, all_full = false;
  DevBuf<MeasDesc> d_meas;
  DevBuf<double> d_times, d_vals, d_uncs, d_profiles, d_irf, d_scratch, d_ladder_T, d_ladder_out, d_ladder_sum, d_hist;
  double* h_ladder_sum = nullptr;      // pinned staging of the per-chain ladder rows
  int* h_nsteps = nullptr;
  size_t h_ladder_cap = 0, h_nsteps_cap = 0;
  int n_ladder = 0;
  bool ladder_valid = false;
  bool any_irf = false, have_irf = false;
  size_t max_nrs = 0, max_nt = 0;
  int irf_rows_needed = 0;
  DevBuf<double> d_params, d_aux, d_logll, d_curves;
  DevBuf<int> d_status, d_nsteps, d_counter, d_order, d_defer, d_queue;
  int queue_n = 0;           // trajectories the explicit queue order is for (0: none)
  int n_sets = 0;
  bool curves_valid = false;
  DevBuf<double> d_fit;
  bool fit_valid = false;
  float last_ms = 0.f;
  int64_t launches = 0;
};

namespace {

// Runs one launch plan: residency, grid, per-slot buffers, then the kernel and (unless
// TRPL_OPT_NO_EXPLICIT) the explicit second pass over the trajectories it deferred.
int run_plan(trpl_handle* h, KernelArgs a, const LaunchPlan& p, const char* what) {
  if (p.smem > (size_t)h->prop.sharedMemPerBlockOptin) return fail("trajectory state does not fit in shared memory");
  const bool two_pass = p.explicit_kernel && !(a.opt.flags & OPT_NO_EXPLICIT);
  if (p.smem > 0) {
    // the occupancy calculator assumes the function's current carve-out: ask for the largest one
    // first, or a small shared-memory request is judged against a small default carve-out
    for (const void* k : {p.kernel, p.explicit_kernel}) {
      if (!k) continue;
      CU(cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
      CU(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem));
    }
  }
  int per_sm = 0;
  CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, p.kernel, p.block, p.smem));
  // CTAs resident on an SM share its 512 tensor-memory columns (a CTA beyond that would sit in
  // tcgen05.alloc until another one exits).  The occupancy calculator answers 1 for any kernel
  // that allocates tensor memory, so residency is computed here: registers and shared memory
  // (launch bounds), capped by the tensor-memory columns.
  if (per_sm >= 1 && p.tm_cols > 0) {
    const int by_smem = (int)((size_t)h->prop.sharedMemPerMultiprocessor / (p.smem + 1024 + 16));
    per_sm = std::min({CTAS_PER_SM * WARPS_PER_CTA / (p.block / 32), by_smem, 512 / p.tm_cols});
  }
  if (per_sm < 1) return fail(std::string(what) + " does not fit on an SM");
  const int grid = std::max(1, std::min(h->prop.multiProcessorCount * per_sm,
                                        (a.n_traj + p.traj_per_cta - 1) / p.traj_per_cta));
  if (getenv("TRPL_DEBUG")) {
    cudaFuncAttributes fa;
    CU(cudaFuncGetAttributes(&fa, p.kernel));
    fprintf(stderr, "[trpl] launch %s, model=%d: %d threads/CTA, %d trajectories/CTA, %zu B dynamic + %zu B static smem/CTA, "
            "%d TMEM columns/CTA, %d CTAs/SM, grid %d\n", what, h->model, p.block, p.traj_per_cta, p.smem,
            fa.sharedSizeBytes, p.tm_cols, per_sm, grid);
  }
  a.slots_per_cta = p.traj_per_cta;
  if (a.scratch_stride > 0) {
    CU(h->d_scratch.reserve((size_t)grid * p.traj_per_cta * a.scratch_stride));
    a.scratch = h->d_scratch.p;
  }
  CU(h->d_hist.reserve((size_t)grid * p.traj_per_cta * 3 * HIST_CAP));
  a.hist = h->d_hist.p;
  CU(cudaMemsetAsync(h->d_counter.p, 0, 4 * sizeof(int), h->stream));
  a.defer_list = nullptr; a.defer_count = h->d_counter.p + 2;
  if (two_pass) {
    CU(h->d_defer.reserve(a.n_traj));
    a.defer_list = h->d_defer.p;
  }
  void* args[] = {&a};
  CU(cudaEventRecord(h->ev0, h->stream));
  for (const void* k : {p.kernel, two_pass ? p.explicit_kernel : nullptr}) {
    if (!k) continue;
    CU(cudaLaunchKernel(k, grid, p.block, args, p.smem, h->stream));
    h->launches += 1;
  }
  if (a.fit) {
    KernelArgs f = a;
    f.slots_per_cta = 1;
    void* fargs[] = {&f};
    CU(cudaLaunchKernel((const void*)trpl_fit_kernel, grid * p.traj_per_cta, 32, fargs, 0, h->stream));
    h->launches += 1;
  }
  CU(cudaEventRecord(h->ev1, h->stream));
  return 0;
}

// One warp per trajectory: at most four warps per CTA (one per tensor-memory lane quarter), fewer if
// their shared-memory slices do not fit the 227 KB of one CTA (the larger grids).
template <int NPL, int MODEL, bool FULL>
int launch(trpl_handle* h, const KernelArgs& a) {
  typedef Slots<NPL, MODEL> SL;
  int wpc = WARPS_PER_CTA;
  while (wpc > 1 && (size_t)wpc * SL::BYTES > (size_t)h->prop.sharedMemPerBlockOptin) --wpc;
  const LaunchPlan p{(const void*)trpl_forward_kernel<NPL, MODEL, FULL>, (const void*)trpl_explicit_kernel<NPL, MODEL, FULL>,
                     32 * wpc, (size_t)wpc * SL::BYTES, TmCta<SL>::COLS, wpc};
  return run_plan(h, a, p, "trajectory kernel");
}

// Grids of 129..256 / 257..512 nodes: a team of two / four warps per trajectory, compiled in
// team_kernels.cu / team4_kernels.cu against the team vocabularies of simt.h (4 nodes per lane on 64 /
// 128 lanes).  Same queue, same arguments, same per-trajectory scratch as launch<>; a CTA of four
// warps holds two trajectories, or one.  Each unit hands out its plan and its sizeof(KernelArgs).
extern "C" size_t trpl_team_plan(int model, int full, LaunchPlan* out);
extern "C" size_t trpl_team4_plan(int model, int full, LaunchPlan* out);

int launch_team(trpl_handle* h, const KernelArgs& a, int team_warps) {
  LaunchPlan p;
  const int full = (h->all_full && h->max_nx == 128 * team_warps) ? 1 : 0;
  if ((team_warps == 4 ? trpl_team4_plan : trpl_team_plan)(h->model, full, &p) != sizeof(KernelArgs))
    return fail("the team kernel unit was built with another KernelArgs layout");
  return run_plan(h, a, p, "team kernel");
}

// CTA-per-trajectory launch (TRPL_OPT_CTA_PER_TRAJ): 'std' model, every measurement on 128 nodes
int launch_cta(trpl_handle* h, const KernelArgs& a) {
  if (h->model != TRPL_MODEL_STD || !h->all_full || h->max_nx != cta::NX)
    return fail("TRPL_OPT_CTA_PER_TRAJ: this instantiation exists for the 'std' model with nx = 128 on every measurement");
  // static shared memory only; one step log / scratch slice per CTA (warp 0 runs the emission)
  return run_plan(h, a, LaunchPlan{(const void*)trpl_cta_kernel, nullptr, cta::NX, 0, 0, 1}, "CTA-per-trajectory kernel");
}

// TRPL_OPT_EXTRAPOLATION: the order-6 extrapolation integrator, one warp per trajectory or (with
// TRPL_OPT_CTA_PER_TRAJ) one CTA per trajectory.  'std' or 'traps' model, every measurement on 128
// nodes.
template <int MODEL>
int launch_seulex_model(trpl_handle* h, const KernelArgs& a, bool cooperative) {
  typedef Slots<4, MODEL> SL;
  const LaunchPlan p{cooperative ? (const void*)trpl_seulex_cta_kernel<4, MODEL, true> : (const void*)trpl_seulex_kernel<4, MODEL, true>,
                     nullptr, 32 * WARPS_PER_CTA,
                     (size_t)WARPS_PER_CTA * SL::BYTES + (cooperative ? (size_t)SeulexXch<4, MODEL>::BYTES : 0),
                     TmCta<SL>::COLS, cooperative ? 1 : WARPS_PER_CTA};
  return run_plan(h, a, p, "extrapolation kernel");
}

int launch_seulex(trpl_handle* h, const KernelArgs& a, bool cooperative) {
  if (!h->all_full || h->max_nx != 128)
    return fail("TRPL_OPT_EXTRAPOLATION: this integrator is built for the 'std' and 'traps' models with nx = 128 on every measurement");
  if (h->model == TRPL_MODEL_STD) return launch_seulex_model<MODEL_STD>(h, a, cooperative);
#ifdef TRPL_DEV_HEADLINE_ONLY
  return fail("this developer build only holds the 'std' model");
#else
  return launch_seulex_model<MODEL_TRAPS>(h, a, cooperative);
#endif
}

template <int MODEL>
int launch_npl(trpl_handle* h, const KernelArgs& a) {
  const int nx = h->max_nx;
#ifdef TRPL_DEV_NX256_ONLY      // developer builds of tuning variants: the nx = 129..512 kernels only
  if (nx > 128 && nx <= 512) return launch_team(h, a, nx <= 256 ? 2 : 4);
  return fail("this developer build only holds the team instantiations (nx > 128)");
#else
  // more than 128 nodes: two or four warps per trajectory (team_kernels.cu, team4_kernels.cu)
  if (nx > 128 && nx <= 512) return launch_team(h, a, nx <= 256 ? 2 : 4);
  // the padding-free instantiation exists for the headline grid (nx = 128)
  if (h->all_full && nx == 128) return launch<4, MODEL, true>(h, a);
#ifdef TRPL_DEV_HEADLINE_ONLY   // developer builds of tuning variants: compile one instantiation only
  return fail("this developer build only holds the nx=128 instantiation");
#else
  if (nx <= 32) return launch<1, MODEL, false>(h, a);
  if (nx <= 64) return launch<2, MODEL, false>(h, a);
  if (nx <= 128) return launch<4, MODEL, false>(h, a);
  return fail("nx > 512 is not supported by this build");
#endif
#endif
}

}  // namespace

extern "C" {

const char* trpl_last_error(void) { return g_err.c_str(); }
int trpl_abi_version(void) { return TRPL_ABI_VERSION; }

int trpl_create(int device, trpl_handle** out) {
  if (!out) return fail("trpl_create: out is NULL");
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n <= 0)
    return fail(std::string("no CUDA device available (") + cudaGetErrorString(e) +
                "); metrotrpl_b200 has no CPU fallback");
  if (device < 0 || device >= n) return fail("trpl_create: bad device index");
  CU(cudaSetDevice(device));
  trpl_handle* h = new trpl_handle();
  h->device = device;
  CU(cudaGetDeviceProperties(&h->prop, device));
  CU(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
  CU(cudaEventCreate(&h->ev0));
  CU(cudaEventCreate(&h->ev1));
  CU(cudaEventCreate(&h->tm0));
  CU(cudaEventCreate(&h->tm1));
  CU(h->d_counter.reserve(4));
  *out = h;
  return 0;
}

void trpl_destroy(trpl_handle* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  cudaStreamSynchronize(h->stream);
  cudaEventDestroy(h->ev0);
  cudaEventDestroy(h->ev1);
  cudaEventDestroy(h->tm0);
  cudaEventDestroy(h->tm1);
  cudaStreamDestroy(h->stream);
  if (h->h_ladder_sum) cudaFreeHost(h->h_ladder_sum);
  if (h->h_nsteps) cudaFreeHost(h->h_nsteps);
  delete h;
}

int trpl_device_info(trpl_handle* h, int32_t* sm_count, int32_t* sm_clock_khz, char* name, int32_t name_len) {
  if (!h) return fail("null handle");
  if (sm_count) *sm_count = h->prop.multiProcessorCount;
  if (sm_clock_khz) {
    int khz = 0;
    cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, h->device);
    *sm_clock_khz = khz;
  }
  if (name && name_len > 0) { strncpy(name, h->prop.name, name_len - 1); name[name_len - 1] = 0; }
  return 0;
}

int trpl_set_problem(trpl_handle* h, int32_t model, int32_t n_meas, const trpl_meas_desc* meas,
                     int32_t n_times_total, const double* times, const double* vals,
                     const double* uncs, int32_t n_profile_total, const double* profiles) {
  if (!h) return fail("null handle");
  if (model != TRPL_MODEL_STD && model != TRPL_MODEL_TRAPS) return fail("Invalid model");
  if (n_meas < 1 || !meas || !times || n_times_total < 1) return fail("trpl_set_problem: empty problem");
  int max_nx = 0;
  for (int i = 0; i < n_meas; ++i) {
    const trpl_meas_desc& m = meas[i];
    if (m.nx < 2 || m.nx > 512) return fail("nx must be in 2..512");
    if (m.n_t < 1 || m.t_off < 0 || m.t_off + m.n_t > n_times_total) return fail("bad time slice");
    if (times[m.t_off] != 0.0) return fail("Grid error - times must start at t=0");   // sim_utils.py:271-272
    for (int k = 1; k < m.n_t; ++k)
      if (!(times[m.t_off + k] > times[m.t_off + k - 1])) return fail("measurement times must be strictly ascending");
    if (m.meas_type != TRPL_MEAS_TRPL && m.meas_type != TRPL_MEAS_TRTS) return fail("TRTS or TRPL only");
    if (m.ini_mode == TRPL_INI_DENSITY) {
      if (!profiles || m.prof_off < 0 || m.prof_off + m.nx > n_profile_total)
        return fail("density mode needs nx initial densities per measurement");
    } else if (m.ini_mode != TRPL_INI_FLUENCE) {
      return fail("Invalid ini_mode - must be 'density' or 'fluence'");
    }
    if (!(m.thickness > 0)) return fail("thickness must be positive");
    if (m.irf_nk < 0 || (m.irf_nk > 0 && !(m.irf_dt > 0))) return fail("bad IRF descriptor");
    if (!(m.min_y >= 0)) return fail("min_y must be non-negative");
    if (m.nx > max_nx) max_nx = m.nx;
  }
  // all measurements of one launch share the nodes-per-lane template: nx must fit 32*NPL and
  // exceed NPL so that the two contacts sit on different lanes
  // (more than 128 nodes: still 4 per lane, on the 64 or 128 lanes of a team)
  const int npl = max_nx <= 32 ? 1 : max_nx <= 64 ? 2 : 4;
  for (int i = 0; i < n_meas; ++i)
    if (meas[i].nx <= npl) return fail("mixed nx: smallest nx must exceed the nodes per lane of the largest grid (1, 2 or 4)");
  CU(cudaSetDevice(h->device));
  CU(h->d_meas.reserve(n_meas));
  CU(h->d_times.reserve(n_times_total));
  CU(cudaMemcpyAsync(h->d_meas.p, meas, sizeof(MeasDesc) * n_meas, cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemcpyAsync(h->d_times.p, times, sizeof(double) * n_times_total, cudaMemcpyHostToDevice, h->stream));
  h->have_vals = vals && uncs;
  if (h->have_vals) {
    CU(h->d_vals.reserve(n_times_total));
    CU(h->d_uncs.reserve(n_times_total));
    CU(cudaMemcpyAsync(h->d_vals.p, vals, sizeof(double) * n_times_total, cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(h->d_uncs.p, uncs, sizeof(double) * n_times_total, cudaMemcpyHostToDevice, h->stream));
  }
  h->have_profiles = profiles && n_profile_total > 0;
  if (h->have_profiles) {
    CU(h->d_profiles.reserve(n_profile_total));
    CU(cudaMemcpyAsync(h->d_profiles.p, profiles, sizeof(double) * n_profile_total, cudaMemcpyHostToDevice, h->stream));
  }
  CU(cudaStreamSynchronize(h->stream));
  {
    // static cost proxy: thicker films and stronger excitation take more integrator steps
    std::vector<std::pair<double, int>> cost(n_meas);
    for (int i = 0; i < n_meas; ++i) {
      const trpl_meas_desc& m = meas[i];
      double amp = m.ini_a;
      if (m.ini_mode == TRPL_INI_DENSITY) { amp = 0; for (int x = 0; x < m.nx; ++x) amp = std::max(amp, profiles[m.prof_off + x]); }
      cost[i] = {-(m.thickness * (double)m.n_t * (1.0 + 0.05 * log10(std::max(amp, 1.0)))), i};
    }
    std::sort(cost.begin(), cost.end());
    std::vector<int> order(n_meas);
    for (int i = 0; i < n_meas; ++i) order[i] = cost[i].second;
    CU(h->d_order.reserve(n_meas));
    CU(cudaMemcpyAsync(h->d_order.p, order.data(), sizeof(int) * n_meas, cudaMemcpyHostToDevice, h->stream));
    CU(cudaStreamSynchronize(h->stream));
  }
  h->any_irf = false; h->have_irf = false; h->max_nrs = 0; h->max_nt = 0; h->irf_rows_needed = 0;
  for (int i = 0; i < n_meas; ++i) {
    const trpl_meas_desc& m = meas[i];
    if ((size_t)m.n_t > h->max_nt) h->max_nt = m.n_t;
    if (m.irf_nk > 0) {
      h->any_irf = true;
      const size_t n_rs = irf_resample_count(times[m.t_off + m.n_t - 1], m.irf_dt);
      if (n_rs > h->max_nrs) h->max_nrs = n_rs;
      if (m.irf_off + m.irf_nk > h->irf_rows_needed) h->irf_rows_needed = m.irf_off + m.irf_nk;
    }
  }
  h->model = model; h->n_meas = n_meas; h->n_times_total = n_times_total; h->max_nx = max_nx;
  h->queue_n = 0;
  h->all_full = true;
  for (int i = 0; i < n_meas; ++i) if (meas[i].nx != max_nx) h->all_full = false;
  return 0;
}

int trpl_set_irf(trpl_handle* h, int32_t n_rows_total, const double* moments) {
  if (!h || !moments || n_rows_total < 1) return fail("trpl_set_irf: bad arguments");
  if (n_rows_total < h->irf_rows_needed) return fail("trpl_set_irf: table shorter than the measurement descriptors need");
  CU(cudaSetDevice(h->device));
  CU(h->d_irf.reserve((size_t)n_rows_total * 3));
  CU(cudaMemcpyAsync(h->d_irf.p, moments, sizeof(double) * 3 * n_rows_total, cudaMemcpyHostToDevice, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  h->have_irf = true;
  return 0;
}

int trpl_set_queue_order(trpl_handle* h, int32_t n_traj, const int32_t* order) {
  if (!h) return fail("null handle");
  if (n_traj <= 0 || !order) { h->queue_n = 0; return 0; }
  std::vector<char> seen(n_traj, 0);
  for (int i = 0; i < n_traj; ++i) {
    const int t = order[i];
    if (t < 0 || t >= n_traj || seen[t]) return fail("trpl_set_queue_order: order is not a permutation of [0, n_traj)");
    seen[t] = 1;
  }
  CU(cudaSetDevice(h->device));
  CU(h->d_queue.reserve(n_traj));
  // pageable source: the runtime stages it before returning, and the copy is ordered before the
  // next launch on the same stream - no host synchronisation needed
  CU(cudaMemcpyAsync(h->d_queue.p, order, sizeof(int) * n_traj, cudaMemcpyHostToDevice, h->stream));
  h->queue_n = n_traj;
  return 0;
}

int trpl_set_ladder(trpl_handle* h, int32_t n_temps, const double* temps) {
  if (!h || n_temps < 1 || !temps) return fail("trpl_set_ladder: bad arguments");
  CU(cudaSetDevice(h->device));
  CU(h->d_ladder_T.reserve(n_temps));
  CU(cudaMemcpyAsync(h->d_ladder_T.p, temps, sizeof(double) * n_temps, cudaMemcpyHostToDevice, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  h->n_ladder = n_temps;
  return 0;
}

int trpl_download_ladder(trpl_handle* h, double* out) {
  if (!h || !out) return fail("null argument");
  if (!h->ladder_valid) return fail("the last run did not produce ladder likelihoods");
  CU(cudaSetDevice(h->device));
  CU(cudaMemcpyAsync(out, h->d_ladder_out.p, sizeof(double) * (size_t)h->n_sets * h->n_meas * h->n_ladder,
                     cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return 0;
}

static int ladder_sums_launch(trpl_handle* h) {
  if (!h->ladder_valid) return fail("the last run did not produce ladder likelihoods");
  CU(cudaSetDevice(h->device));
  const int n = h->n_sets * h->n_ladder;
  CU(h->d_ladder_sum.reserve(n));
  ladder_sum_kernel<<<(n + 255) / 256, 256, 0, h->stream>>>(h->d_ladder_out.p, h->d_ladder_sum.p, h->n_sets,
                                                             h->n_meas, h->n_ladder);
  CU(cudaGetLastError());
  h->launches += 1;
  return 0;
}

int trpl_ladder_sums_resident(trpl_handle* h, const double** dev_rows, int32_t* n_sets, int32_t* n_temps) {
  if (!h || !dev_rows) return fail("null argument");
  if (int r = ladder_sums_launch(h)) return r;
  CU(cudaStreamSynchronize(h->stream));
  *dev_rows = h->d_ladder_sum.p;
  if (n_sets) *n_sets = h->n_sets;
  if (n_temps) *n_temps = h->n_ladder;
  return 0;
}

int trpl_download_ladder_sums(trpl_handle* h, double* rows, int32_t* nsteps) {
  if (!h || !rows) return fail("null argument");
  if (int r = ladder_sums_launch(h)) return r;
  const size_t n = (size_t)h->n_sets * h->n_ladder, n_traj = (size_t)h->n_sets * h->n_meas;
  // pinned staging: the copies are truly asynchronous and one synchronisation serves both
  if (n > h->h_ladder_cap) {
    if (h->h_ladder_sum) cudaFreeHost(h->h_ladder_sum);
    CU(cudaMallocHost(&h->h_ladder_sum, n * sizeof(double)));
    h->h_ladder_cap = n;
  }
  if (nsteps && 2 * n_traj > h->h_nsteps_cap) {
    if (h->h_nsteps) cudaFreeHost(h->h_nsteps);
    CU(cudaMallocHost(&h->h_nsteps, 2 * n_traj * sizeof(int)));
    h->h_nsteps_cap = 2 * n_traj;
  }
  CU(cudaMemcpyAsync(h->h_ladder_sum, h->d_ladder_sum.p, n * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  if (nsteps) CU(cudaMemcpyAsync(h->h_nsteps, h->d_nsteps.p, 2 * n_traj * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  memcpy(rows, h->h_ladder_sum, n * sizeof(double));
  if (nsteps) memcpy(nsteps, h->h_nsteps, 2 * n_traj * sizeof(int));
  return 0;
}

int trpl_download_nsteps(trpl_handle* h, int32_t* nsteps) {
  if (!h || !nsteps) return fail("null argument");
  CU(cudaSetDevice(h->device));
  CU(cudaMemcpyAsync(nsteps, h->d_nsteps.p, sizeof(int) * 2 * (size_t)h->n_sets * h->n_meas, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return 0;
}

int trpl_upload_batch(trpl_handle* h, int32_t n_sets, const double* params, const double* aux) {
  if (!h) return fail("null handle");
  if (h->n_meas < 1) return fail("trpl_set_problem has not been called");
  if (n_sets < 1 || !params || !aux) return fail("empty batch");
  CU(cudaSetDevice(h->device));
  const size_t n_traj = (size_t)n_sets * h->n_meas;
  CU(h->d_params.reserve((size_t)n_sets * TRPL_NPARAM));
  CU(h->d_aux.reserve(n_traj * TRPL_NAUX));
  CU(h->d_logll.reserve(n_traj * 3));
  CU(h->d_status.reserve(n_traj));
  CU(h->d_nsteps.reserve(n_traj * 2));
  CU(cudaMemcpyAsync(h->d_params.p, params, sizeof(double) * n_sets * TRPL_NPARAM, cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemcpyAsync(h->d_aux.p, aux, sizeof(double) * n_traj * TRPL_NAUX, cudaMemcpyHostToDevice, h->stream));
  h->n_sets = n_sets;
  return 0;
}

int trpl_run_resident(trpl_handle* h, const trpl_solver_opts* opts, int32_t want_curves) {
  if (!h || !opts) return fail("null argument");
  if (h->n_sets < 1) return fail("no batch uploaded");
  if (!(opts->rtol > 0) || !(opts->atol >= 0) || opts->max_steps < 1) return fail("bad solver options");
  h->fit_valid = false;
  RunPlan p;
  const ProblemFacts pf{h->have_vals, h->any_irf, h->have_irf, h->n_ladder, h->max_nrs, h->max_nt};
  if (const char* why = plan_run(pf, opts->flags, want_curves != 0, p)) return fail(why);
  CU(cudaSetDevice(h->device));
  if (p.curves) CU(h->d_curves.reserve((size_t)h->n_sets * h->n_times_total));
  h->curves_valid = p.curves;
  h->ladder_valid = false;
  if (p.ladder) CU(h->d_ladder_out.reserve((size_t)h->n_sets * h->n_meas * h->n_ladder));
  h->ladder_valid = p.ladder;
  if (p.fit) CU(h->d_fit.reserve((size_t)h->n_sets * h->n_times_total));
  h->fit_valid = p.fit;
  KernelArgs a;
  a.params = h->d_params.p; a.aux = h->d_aux.p; a.meas = h->d_meas.p; a.times = h->d_times.p;
  a.vals = h->have_vals ? h->d_vals.p : nullptr; a.uncs = h->have_vals ? h->d_uncs.p : nullptr;
  a.profiles = h->have_profiles ? h->d_profiles.p : nullptr;
  a.logll = h->d_logll.p; a.status = h->d_status.p; a.nsteps = h->d_nsteps.p;
  p.set_args(a, h->d_curves.p, h->d_irf.p, h->d_ladder_T.p, h->d_ladder_out.p, h->n_ladder, h->d_fit.p);
  a.counter = h->d_counter.p;
  a.meas_order = h->d_order.p;
  a.queue = (h->queue_n > 0 && h->queue_n == h->n_sets * h->n_meas) ? h->d_queue.p : nullptr;
  a.n_traj = h->n_sets * h->n_meas; a.n_meas = h->n_meas; a.n_times_total = h->n_times_total;
  memcpy(&a.opt, opts, sizeof(SolverOpts));
  if (opts->flags & TRPL_OPT_EXTRAPOLATION) return launch_seulex(h, a, (opts->flags & TRPL_OPT_CTA_PER_TRAJ) != 0);
  if (opts->flags & TRPL_OPT_CTA_PER_TRAJ) return launch_cta(h, a);
  if (h->model == TRPL_MODEL_STD) return launch_npl<MODEL_STD>(h, a);
#ifdef TRPL_DEV_HEADLINE_ONLY
  return fail("this developer build only holds the 'std' model");
#else
  return launch_npl<MODEL_TRAPS>(h, a);
#endif
}

int trpl_download_fit(trpl_handle* h, double* fit) {
  if (!h || !fit) return fail("null argument");
  if (!h->fit_valid) return fail("the last run did not produce fitted curves (run with TRPL_OPT_FIT)");
  CU(cudaSetDevice(h->device));
  CU(cudaMemcpyAsync(fit, h->d_fit.p, sizeof(double) * (size_t)h->n_sets * h->n_times_total, cudaMemcpyDeviceToHost,
                     h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return 0;
}

int trpl_download_results(trpl_handle* h, double* logll, int32_t* status, int32_t* nsteps, double* curves) {
  if (!h) return fail("null handle");
  CU(cudaSetDevice(h->device));
  const size_t n_traj = (size_t)h->n_sets * h->n_meas;
  if (logll) CU(cudaMemcpyAsync(logll, h->d_logll.p, sizeof(double) * n_traj * 3, cudaMemcpyDeviceToHost, h->stream));
  if (status) CU(cudaMemcpyAsync(status, h->d_status.p, sizeof(int) * n_traj, cudaMemcpyDeviceToHost, h->stream));
  if (nsteps) CU(cudaMemcpyAsync(nsteps, h->d_nsteps.p, sizeof(int) * n_traj * 2, cudaMemcpyDeviceToHost, h->stream));
  if (curves) {
    if (!h->curves_valid) return fail("curves were not produced by the last run");
    CU(cudaMemcpyAsync(curves, h->d_curves.p, sizeof(double) * h->n_sets * h->n_times_total, cudaMemcpyDeviceToHost, h->stream));
  }
  CU(cudaStreamSynchronize(h->stream));
  CU(cudaEventElapsedTime(&h->last_ms, h->ev0, h->ev1));
  return 0;
}

int trpl_loglik_batch(trpl_handle* h, int32_t n_sets, const double* params, const double* aux,
                      const trpl_solver_opts* opts, double* logll, int32_t* status, int32_t* nsteps,
                      double* curves) {
  if (int r = trpl_upload_batch(h, n_sets, params, aux)) return r;
  if (int r = trpl_run_resident(h, opts, curves != nullptr)) return r;
  return trpl_download_results(h, logll, status, nsteps, curves);
}

int trpl_solve_batch(trpl_handle* h, int32_t n_sets, const double* params, const double* aux,
                     const trpl_solver_opts* opts, double* curves, int32_t* status, int32_t* nsteps) {
  if (!opts || !curves) return fail("null argument");
  trpl_solver_opts o = *opts;
  o.flags |= TRPL_OPT_NO_LIKELIHOOD;
  if (int r = trpl_upload_batch(h, n_sets, params, aux)) return r;
  if (int r = trpl_run_resident(h, &o, 1)) return r;
  return trpl_download_results(h, nullptr, status, nsteps, curves);
}

int trpl_last_kernel_ms(trpl_handle* h, float* ms) {
  if (!h || !ms) return fail("null argument");
  CU(cudaSetDevice(h->device));
  CU(cudaEventSynchronize(h->ev1));
  CU(cudaEventElapsedTime(&h->last_ms, h->ev0, h->ev1));
  *ms = h->last_ms;
  return 0;
}

int64_t trpl_launch_count(trpl_handle* h) { return h ? h->launches : 0; }

int trpl_synchronize(trpl_handle* h) {
  if (!h) return fail("null handle");
  CU(cudaSetDevice(h->device));
  CU(cudaStreamSynchronize(h->stream));
  return 0;
}

int trpl_timer_begin(trpl_handle* h) {
  if (!h) return fail("null handle");
  CU(cudaSetDevice(h->device));
  CU(cudaStreamSynchronize(h->stream));
  CU(cudaEventRecord(h->tm0, h->stream));
  return 0;
}

int trpl_timer_end(trpl_handle* h, float* ms) {
  if (!h || !ms) return fail("null argument");
  CU(cudaSetDevice(h->device));
  CU(cudaEventRecord(h->tm1, h->stream));
  CU(cudaEventSynchronize(h->tm1));
  CU(cudaEventElapsedTime(ms, h->tm0, h->tm1));
  return 0;
}

int trpl_flush_l2(trpl_handle* h) {
  if (!h) return fail("null handle");
  CU(cudaSetDevice(h->device));
  const size_t bytes = (size_t)256 << 20;
  CU(h->d_flush.reserve(bytes));
  CU(cudaMemsetAsync(h->d_flush.p, 1, bytes, h->stream));
  return 0;
}

int trpl_make_trial_moves(int32_t n_chains, int32_t n_par, const double* cur, const double* moves,
                          const uint8_t* do_log, const uint8_t* active, const double* lo, const double* hi,
                          int32_t idx_p0, int32_t idx_n0, int32_t idx_taun, int32_t idx_taup,
                          int32_t hard_bounds, int32_t max_tries, const uint64_t pcg_state[2],
                          const uint64_t pcg_inc[2], double* proposals, double* u, int64_t* n_draws,
                          int32_t* n_failed, uint32_t* fail_masks, int32_t idx_mun, int32_t idx_mup,
                          double ambi_lo, double ambi_hi, const double* ambi_u, int32_t n_ambi_u,
                          int32_t* n_ambi_used, double* mu_arg) {
  if (n_chains < 1 || n_par < 1 || n_par > 30) return fail("trpl_make_trial_moves: 1..30 parameters");
  if (!cur || !moves || !do_log || !active || !lo || !hi || !pcg_state || !pcg_inc || !proposals || !u ||
      !n_draws || !n_failed || !fail_masks || max_tries < 1)
    return fail("trpl_make_trial_moves: bad arguments");
  if (idx_mun >= 0 && (idx_mup < 0 || idx_mun >= n_par || idx_mup >= n_par || !ambi_u || n_ambi_u < 1 || !mu_arg))
    return fail("trpl_make_trial_moves: the mobility constraint needs both indices and pre-drawn uniforms");
  const int rc = trpl_host::make_trial_moves(n_chains, n_par, cur, moves, do_log, active, lo, hi, idx_p0, idx_n0,
                                             idx_taun, idx_taup, hard_bounds, max_tries, pcg_state, pcg_inc,
                                             proposals, u, n_draws, n_failed, fail_masks, TRPL_MAX_LOGGED_FAILS,
                                             idx_mun, idx_mup, ambi_lo, ambi_hi, ambi_u, n_ambi_u, n_ambi_used, mu_arg);
  if (rc == 2) return fail("trpl_make_trial_moves: ran out of pre-drawn uniforms for the mobility constraint");
  return rc;
}

int trpl_fp64_peak_probe(trpl_handle* h, int32_t iters, double* tflops, float* ms_out) {
  if (!h || !tflops) return fail("null argument");
  CU(cudaSetDevice(h->device));
  const int threads = 256, blocks = h->prop.multiProcessorCount * 8;
  DevBuf<double> sink;
  CU(sink.reserve((size_t)threads * blocks));
  fp64_probe_kernel<<<blocks, threads, 0, h->stream>>>(sink.p, 1000, 1.0);   // warm-up
  CU(cudaEventRecord(h->ev0, h->stream));
  fp64_probe_kernel<<<blocks, threads, 0, h->stream>>>(sink.p, iters, 1.0);
  CU(cudaGetLastError());
  CU(cudaEventRecord(h->ev1, h->stream));
  CU(cudaEventSynchronize(h->ev1));
  float ms = 0.f;
  CU(cudaEventElapsedTime(&ms, h->ev0, h->ev1));
  h->launches += 2;
  const double flops = 2.0 * 8.0 * (double)iters * threads * blocks;
  *tflops = flops / (ms * 1e-3) / 1e12;
  if (ms_out) *ms_out = ms;
  return 0;
}

}  // extern "C"
