// simt.h - the one-warp SIMT vocabulary the trajectory integrator is written in.
//
// The integrator (trajectory.h and the headers it includes) is written once against this
// vocabulary: `real` is "one double per lane", `mask` is "one predicate per lane", control flow
// is warp-uniform, and all cross-lane traffic goes through shfl_* / warp_* / ballot.
//
//   * Device build (nvcc, sm_100a): real == double, every function is a forced-inline wrapper
//     around the warp intrinsic it names.  This is the product.
//   * Host lock-step build (-DTRPL_HOST_EMU, g++): real is a 32-wide array with overloaded
//     arithmetic, shuffles are permutations.  It exists so tests/ can run the very same
//     integrator source on a CPU-only box; it is compiled only by tests/emu and is never
//     reachable from the metrotrpl_b200 package.
#pragma once
#include <math.h>
#include <stdint.h>

// TRPL_TEAM: warps that integrate one trajectory together.  1 (default): the one-warp vocabulary
// described above.  2 or 4: a TEAM of that many warps is the "wide warp" - 64 or 128 lanes, lane_id()
// 0..LANES-1 - and every cross-lane primitive spans all its warps: shuffles between neighbours hand
// the one value that crosses each warp boundary through a shared-memory mailbox, reductions combine
// the warps' partials there in a fixed order, warp_sync() is a named barrier of the team's threads.
// The integrator source is the same; team_kernels.cu / team4_kernels.cu compile it again with this
// vocabulary for the grids of 129..256 / 257..512 nodes (4 nodes per lane: the state fits the
// register file, where one warp with 8 or 16 nodes per lane spills).
#ifndef TRPL_TEAM
#define TRPL_TEAM 1
#endif
#if TRPL_TEAM != 1 && TRPL_TEAM != 2 && TRPL_TEAM != 4
#error "TRPL_TEAM must be 1, 2 or 4"
#endif

#if defined(__CUDACC__) && !defined(TRPL_HOST_EMU)
// ------------------------------------------------------------------------------------------
// device
// ------------------------------------------------------------------------------------------
#define TRPL_FN __device__ __forceinline__
#define TRPL_HD __host__ __device__ __forceinline__     // also called by the library's host code
#define TRPL_UNROLL _Pragma("unroll")
#define TRPL_UNROLL4 _Pragma("unroll 4")

namespace simt {
typedef double real;
typedef bool mask;
typedef int ivec;
constexpr unsigned FULL = 0xffffffffu;
constexpr int LANES = 32 * TRPL_TEAM;            // lanes of the (wide) warp that owns a trajectory
constexpr int LOG2_LANES = TRPL_TEAM == 4 ? 7 : TRPL_TEAM == 2 ? 6 : 5;

TRPL_FN ivec lane_id() { return (int)(threadIdx.x & (unsigned)(LANES - 1)); }
TRPL_FN real splat(double x) { return x; }
TRPL_FN double uni(real x) { return x; }                 // x is known to be warp-uniform
#if TRPL_TEAM == 1
typedef unsigned lanebits;                                // one bit per lane (warp_ballot)
TRPL_FN double lane0(real x) { return __shfl_sync(FULL, x, 0); }
TRPL_FN real shfl_up(real x, int d) { return __shfl_up_sync(FULL, x, d); }     // from lane-d (own if out of range)
TRPL_FN real shfl_down(real x, int d) { return __shfl_down_sync(FULL, x, d); } // from lane+d (own if out of range)
TRPL_FN real shfl_idx(real x, int src) { return __shfl_sync(FULL, x, src); }
// batched forms (one exchange in the two-warp vocabulary): N values from the previous / next lane,
// both directions at once, two sums at once
template <int N> TRPL_FN void nbr_up(const real (&x)[N], real (&y)[N]) {
  TRPL_UNROLL for (int i = 0; i < N; ++i) y[i] = __shfl_up_sync(FULL, x[i], 1);
}
template <int N> TRPL_FN void nbr_down(const real (&x)[N], real (&y)[N]) {
  TRPL_UNROLL for (int i = 0; i < N; ++i) y[i] = __shfl_down_sync(FULL, x[i], 1);
}
template <int NU, int ND> TRPL_FN void nbr_both(const real (&xu)[NU], real (&yu)[NU], const real (&xd)[ND], real (&yd)[ND]) {
  nbr_up<NU>(xu, yu); nbr_down<ND>(xd, yd);
}
#else
// ---- team of W = TRPL_TEAM warps: every cross-lane primitive is  [write mailbox] -> team barrier -> [read] ----
// One barrier per primitive, no barrier after the read: a mailbox slot may therefore be written
// again only after ANOTHER team primitive (whose barrier every reader has reached) has run in
// between.  Every CALL SITE has a slot of its own (the macros at the end of this file hand out
// __COUNTER__; the kernel units assert that there are at most TEAM_SLOTS sites), so only a site
// that runs twice in a row with no other team primitive in between could collide; the host
// lock-step build runs the same slot numbers and aborts if two consecutive primitives of a
// trajectory share one.  A CTA is always four warps (one per tensor-memory lane quarter): two teams
// of two warps, or one team of four.
#if TRPL_TEAM == 4
typedef unsigned __int128 lanebits;
#else
typedef unsigned long long lanebits;
#endif
constexpr int TEAM_WARPS = TRPL_TEAM;
constexpr int TEAMS_PER_CTA = 4 / TRPL_TEAM;
constexpr int TEAM_SLOTS = 64;
constexpr int TEAM_SLOT_VALUES = 8;                                        // values per warp boundary and slot
constexpr int TEAM_SLOT_DOUBLES = TEAM_SLOT_VALUES * (TEAM_WARPS - 1);     // (reductions use 2 per warp: <= 8)
TRPL_FN unsigned team_index() { return (threadIdx.x / (unsigned)LANES) & (unsigned)(TEAMS_PER_CTA - 1); }
TRPL_FN unsigned team_warp() { return (threadIdx.x >> 5) & (unsigned)(TEAM_WARPS - 1); }   // warp within its team
TRPL_FN double* team_box(int slot) {
  __shared__ double box[TEAMS_PER_CTA][TEAM_SLOTS][TEAM_SLOT_DOUBLES];
  return &box[team_index()][slot][0];
}
TRPL_FN void team_bar() { asm volatile("bar.sync %0, %1;" :: "r"(1 + (int)team_index()), "n"(LANES) : "memory"); }
template <int S> TRPL_FN double lane0_s(real x) {
  volatile double* b = team_box(S);
  if ((threadIdx.x & (unsigned)(LANES - 1)) == 0u) b[0] = x;
  team_bar();
  return b[0];
}
template <int S> TRPL_FN real shfl_idx_s(real x, int src) {
  volatile double* b = team_box(S);
  if ((int)(threadIdx.x & (unsigned)(LANES - 1)) == src) b[0] = x;
  team_bar();
  return b[0];
}
// Neighbour exchanges (distance 1, all the integrator uses): the hardware shuffle inside each warp;
// the value that crosses a warp boundary goes from lane 31 of warp w to lane 0 of warp w+1 (or back)
// through that boundary's part of the slot.  Up to TEAM_SLOT_VALUES values behind ONE barrier.
template <int S, int NU, int ND>
TRPL_FN void nbr_both_s(const real (&xu)[NU], real (&yu)[NU], const real (&xd)[ND], real (&yd)[ND]) {
  static_assert(NU + ND <= TEAM_SLOT_VALUES, "mailbox slot too small");
  volatile double* b = team_box(S);
  const unsigned wl = threadIdx.x & 31u, w = team_warp();
  TRPL_UNROLL for (int i = 0; i < NU; ++i) yu[i] = __shfl_up_sync(FULL, xu[i], 1);
  TRPL_UNROLL for (int i = 0; i < ND; ++i) yd[i] = __shfl_down_sync(FULL, xd[i], 1);
  if (wl == 31u && w + 1u < (unsigned)TEAM_WARPS) { TRPL_UNROLL for (int i = 0; i < NU; ++i) b[w * TEAM_SLOT_VALUES + i] = xu[i]; }
  if (wl == 0u && w > 0u) { TRPL_UNROLL for (int i = 0; i < ND; ++i) b[(w - 1u) * TEAM_SLOT_VALUES + NU + i] = xd[i]; }
  team_bar();
  if (wl == 0u && w > 0u) { TRPL_UNROLL for (int i = 0; i < NU; ++i) yu[i] = b[(w - 1u) * TEAM_SLOT_VALUES + i]; }
  if (wl == 31u && w + 1u < (unsigned)TEAM_WARPS) { TRPL_UNROLL for (int i = 0; i < ND; ++i) yd[i] = b[w * TEAM_SLOT_VALUES + NU + i]; }
}
template <int S, int N> TRPL_FN void nbr_up_s(const real (&x)[N], real (&y)[N]) {
  static_assert(N <= TEAM_SLOT_VALUES, "mailbox slot too small");
  volatile double* b = team_box(S);
  const unsigned wl = threadIdx.x & 31u, w = team_warp();
  TRPL_UNROLL for (int i = 0; i < N; ++i) y[i] = __shfl_up_sync(FULL, x[i], 1);
  if (wl == 31u && w + 1u < (unsigned)TEAM_WARPS) { TRPL_UNROLL for (int i = 0; i < N; ++i) b[w * TEAM_SLOT_VALUES + i] = x[i]; }
  team_bar();
  if (wl == 0u && w > 0u) { TRPL_UNROLL for (int i = 0; i < N; ++i) y[i] = b[(w - 1u) * TEAM_SLOT_VALUES + i]; }
}
template <int S, int N> TRPL_FN void nbr_down_s(const real (&x)[N], real (&y)[N]) {
  static_assert(N <= TEAM_SLOT_VALUES, "mailbox slot too small");
  volatile double* b = team_box(S);
  const unsigned wl = threadIdx.x & 31u, w = team_warp();
  TRPL_UNROLL for (int i = 0; i < N; ++i) y[i] = __shfl_down_sync(FULL, x[i], 1);
  if (wl == 0u && w > 0u) { TRPL_UNROLL for (int i = 0; i < N; ++i) b[(w - 1u) * TEAM_SLOT_VALUES + i] = x[i]; }
  team_bar();
  if (wl == 31u && w + 1u < (unsigned)TEAM_WARPS) { TRPL_UNROLL for (int i = 0; i < N; ++i) y[i] = b[w * TEAM_SLOT_VALUES + i]; }
}
template <int S> TRPL_FN real shfl_up_s(real x, int) {
  const real in[1] = {x}; real out[1];
  nbr_up_s<S, 1>(in, out);
  return out[0];
}
template <int S> TRPL_FN real shfl_down_s(real x, int) {
  const real in[1] = {x}; real out[1];
  nbr_down_s<S, 1>(in, out);
  return out[0];
}
#endif
TRPL_FN real sel(mask m, real a, real b) { return m ? a : b; }
TRPL_FN ivec seli(mask m, ivec a, ivec b) { return m ? a : b; }
TRPL_FN mask mand(mask a, mask b) { return a && b; }
TRPL_FN mask mor(mask a, mask b) { return a || b; }
TRPL_FN mask mnot(mask a) { return !a; }
TRPL_FN mask mconst(bool b) { return b; }
#if TRPL_TEAM == 1
TRPL_FN bool warp_any(mask m) { return __any_sync(FULL, m) != 0; }
TRPL_FN lanebits warp_ballot(mask m) { return __ballot_sync(FULL, m); }
#else
template <int S> TRPL_FN lanebits warp_ballot_s(mask m) {
  volatile double* b = team_box(S);
  const unsigned mine = __ballot_sync(FULL, m);
  if ((threadIdx.x & 31u) == 0u) b[team_warp()] = (double)mine;      // exact: < 2^32
  team_bar();
  lanebits r = 0;
  TRPL_UNROLL for (int w = 0; w < TEAM_WARPS; ++w) r |= (lanebits)(unsigned)b[w] << (32 * w);
  return r;
}
template <int S> TRPL_FN bool warp_any_s(mask m) { return warp_ballot_s<S>(m) != 0u; }
#endif
TRPL_FN mask lane_lt(ivec l, int k) { return l < k; }
// "does any lane near me see m": evaluated per hardware warp, no team barrier.  Only for choosing
// between two code paths that give the same result and contain no cross-lane primitive.
TRPL_FN bool local_any(mask m) { return __any_sync(FULL, m) != 0; }
TRPL_FN real fmadd(real a, real b, real c) { return fma(a, b, c); }
// Reciprocal: hardware seed (MUFU.RCP64H, ~2^-23) + two Newton steps, no special-case slow path.
// Every argument on this path is a finite, normal, non-zero number (densities, determinants of
// diagonally dominated blocks, error scales), so the IEEE corner cases of `1.0 / x` are not needed.
TRPL_FN real rcp(real x) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
  double e = fma(-x, r, 1.0);
  r = fma(r, e, r);
  e = fma(-x, r, 1.0);
  r = fma(r, e, r);
  return r;
}
TRPL_FN real vdiv(real a, real b) { return a / b; }       // IEEE division (cold paths only)
// Reciprocal to ~2^-23 (the hardware seed alone): for quantities that only steer the step size.
TRPL_FN real rcp_approx(real x) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
  return r;
}
// max of two non-NaN values without fmax's NaN bookkeeping (NaN states are detected separately)
TRPL_FN real vmax_fast(real a, real b) { return a > b ? a : b; }
// x^y for the step-size controller (warp-uniform scalars, single precision, x > 0)
TRPL_FN float ctl_powf(float x, float y) { return __powf(x, y); }
TRPL_FN real vabs(real x) { return fabs(x); }
TRPL_FN real vmax(real a, real b) { return fmax(a, b); }
TRPL_FN real vmin(real a, real b) { return fmin(a, b); }
TRPL_FN real vexp(real x) { return exp(x); }
TRPL_FN real vlog(real x) { return log(x); }
TRPL_FN real vlog10(real x) { return log10(x); }
TRPL_FN real vsqrt(real x) { return sqrt(x); }
TRPL_FN mask is_nan(real x) { return x != x; }
#if TRPL_TEAM == 1
TRPL_FN real warp_sum(real x) {
  TRPL_UNROLL for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(FULL, x, o);
  return x;  // bit-identical on every lane (fp add is commutative)
}
TRPL_FN void warp_sum2(real& a, real& b) { a = warp_sum(a); b = warp_sum(b); }
TRPL_FN real warp_max(real x) {
  TRPL_UNROLL for (int o = 16; o > 0; o >>= 1) x = fmax(x, __shfl_xor_sync(FULL, x, o));
  return x;
}
// inclusive prefix sum over lanes (Gauss's law: E-field from the running net charge)
TRPL_FN real warp_scan_incl(real x) {
  const int l = lane_id();
  TRPL_UNROLL for (int o = 1; o < 32; o <<= 1) {
    real y = __shfl_up_sync(FULL, x, o);
    if (l >= o) x += y;
  }
  return x;
}
#else
// reductions: each warp reduces with shuffles, the partials meet in the mailbox and every warp
// combines them in the same order (identical bits on all lanes: control flow stays team-uniform)
TRPL_FN double team_combine_sum(volatile double* b) {
  if constexpr (TEAM_WARPS == 2) return b[0] + b[1]; else return (b[0] + b[1]) + (b[2] + b[3]);
}
template <int S> TRPL_FN real warp_sum_s(real x) {
  volatile double* b = team_box(S);
  TRPL_UNROLL for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(FULL, x, o);
  if ((threadIdx.x & 31u) == 0u) b[team_warp()] = x;
  team_bar();
  return team_combine_sum(b);
}
template <int S> TRPL_FN void warp_sum2_s(real& x, real& y) {
  volatile double* b = team_box(S);
  TRPL_UNROLL for (int o = 16; o > 0; o >>= 1) { x += __shfl_xor_sync(FULL, x, o); y += __shfl_xor_sync(FULL, y, o); }
  if ((threadIdx.x & 31u) == 0u) { const unsigned w = team_warp(); b[w] = x; b[TEAM_WARPS + w] = y; }
  team_bar();
  x = team_combine_sum(b); y = team_combine_sum(b + TEAM_WARPS);
}
template <int S> TRPL_FN real warp_max_s(real x) {
  volatile double* b = team_box(S);
  TRPL_UNROLL for (int o = 16; o > 0; o >>= 1) x = fmax(x, __shfl_xor_sync(FULL, x, o));
  if ((threadIdx.x & 31u) == 0u) b[team_warp()] = x;
  team_bar();
  real r = fmax(b[0], b[1]);
  if constexpr (TEAM_WARPS == 4) r = fmax(r, fmax(b[2], b[3]));
  return r;
}
template <int S> TRPL_FN real warp_min_s(real x) { return -warp_max_s<S>(-x); }
template <int S> TRPL_FN real warp_scan_incl_s(real x) {
  volatile double* b = team_box(S);
  const int l = (int)(threadIdx.x & 31u);
  TRPL_UNROLL for (int o = 1; o < 32; o <<= 1) {
    real y = __shfl_up_sync(FULL, x, o);
    if (l >= o) x += y;
  }
  const unsigned w = team_warp();
  if (l == 31) b[w] = x;                                   // total of this warp
  team_bar();
  // totals of the warps before this one, added up in warp order
  real off = 0.0;
  TRPL_UNROLL for (int k = 0; k + 1 < TEAM_WARPS; ++k) if ((unsigned)k < w) off = (k == 0) ? (real)b[0] : off + b[k];
  if (w > 0u) x += off;
  return x;
}
#endif
TRPL_FN real gather(const double* p, ivec idx, mask m, double other) { return m ? p[idx] : other; }
// p[idx], p[idx+1] in one 128-bit load (p + idx is 16-byte aligned: idx even, p a scratch slice)
TRPL_FN void gather2(const double* p, ivec idx, mask m, double other, real& a, real& b) {
  if (m) { const double2 v = *reinterpret_cast<const double2*>(p + idx); a = v.x; b = v.y; }
  else { a = other; b = other; }
}
TRPL_FN void scatter(double* p, ivec idx, mask m, real v) { if (m) p[idx] = v; }
TRPL_FN ivec iadd(ivec a, int b) { return a + b; }
TRPL_FN ivec imul(ivec a, int b) { return a * b; }
TRPL_FN ivec irsub(int a, ivec b) { return a - b; }
TRPL_FN ivec iaddv(ivec a, ivec b) { return a + b; }
TRPL_FN ivec isubv(ivec a, ivec b) { return a - b; }
TRPL_FN ivec ishr1(ivec a) { return a >> 1; }
TRPL_FN ivec iclamp(ivec a, int lo, int hi) { return a < lo ? lo : (a > hi ? hi : a); }
TRPL_FN ivec isplat(int a) { return a; }
TRPL_FN ivec to_int_floor(real x) { return (int)floor(x); }
#if TRPL_TEAM == 1
TRPL_FN real warp_min(real x) { return -warp_max(-x); }
#endif
TRPL_FN real to_real(ivec a) { return (double)a; }
TRPL_FN ivec lane_minus(int d) { const int l = lane_id(); return l >= d ? l - d : l; }   // own lane if out of range
TRPL_FN ivec lane_plus(int d) { const int l = lane_id(); return l + d < LANES ? l + d : l; }

// Per-warp scratch in shared memory, pair-major: pair p of lane l is the 16-byte word
// base[p*32 + l].  Every access is one 128-bit LDS/STS per lane, conflict-free across the warp.
struct LaneMem {
  double2* base;
  TRPL_FN void ld2(int p, real& a, real& b) const { const double2 v = base[p * LANES + lane_id()]; a = v.x; b = v.y; }
  TRPL_FN void st2(int p, real a, real b) const { base[p * LANES + lane_id()] = make_double2(a, b); }
  // read another lane's pair (lane exchange through shared memory; caller orders with warp_sync)
  TRPL_FN void ld2_from(int p, ivec src, real& a, real& b) const { const double2 v = base[p * LANES + src]; a = v.x; b = v.y; }
  // warp-uniform scalars parked in pair slot p (64 doubles): every lane reads the same word (broadcast)
  TRPL_FN double uld(int p, int i) const { return reinterpret_cast<const double*>(base + p * LANES)[i]; }
  TRPL_FN void ust(int p, int i, double v) const { reinterpret_cast<double*>(base + p * LANES)[i] = v; }
};
#if TRPL_TEAM == 1
TRPL_FN void warp_sync() { __syncwarp(); }
#else
TRPL_FN void warp_sync() { team_bar(); }
#endif

// Per-warp scratch in TENSOR MEMORY (sm_100a TMEM, 128 lanes x 512 columns x 32 bit per SM), used
// as lane-private storage: warp w of a CTA owns TMEM lanes 32*(w%4)..+31, thread l of the warp
// reads and writes only its own lane, and pair p of the warp's slice is the four 32-bit columns
// base+4p..+3 of that lane (tcgen05.ld/st .32x32b).  Nothing here is ever an MMA operand: TMEM is
// simply a second on-chip memory with its own data path (measured 400 B/clk/SM against the
// 128 B/clk/SM of shared memory, tools/proto/tmem_probe.cu), which takes the lane-private traffic
// (stage increments, factor blocks) off the shared-memory pipe.  Loads are asynchronous: issue a
// batch, then wait_ld() before the first use; wait_st() before re-reading what was just stored.
struct LaneTm {
  unsigned base;     // (first lane of this warp's quarter << 16) | first column of its slice
  TRPL_FN void st2(int p, real a, real b) const {
    asm volatile("{\n .reg .b32 t0,t1,t2,t3;\n mov.b64 {t0,t1}, %1;\n mov.b64 {t2,t3}, %2;\n"
                 " tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {t0,t1,t2,t3};\n}"
                 :: "r"(base + 4u * (unsigned)p), "d"(a), "d"(b) : "memory");
  }
  TRPL_FN void ld2(int p, real& a, real& b) const {
    asm volatile("{\n .reg .b32 t0,t1,t2,t3;\n tcgen05.ld.sync.aligned.32x32b.x4.b32 {t0,t1,t2,t3}, [%2];\n"
                 " mov.b64 %0, {t0,t1};\n mov.b64 %1, {t2,t3};\n}"
                 : "=d"(a), "=d"(b) : "r"(base + 4u * (unsigned)p) : "memory");
  }
  // two / four consecutive pairs per instruction.  A tcgen05.ld/st costs the tensor-memory pipe
  // about the same whether it moves 4 or 16 columns (measured: ~5.5 clk per instruction per SM), so
  // everything is laid out to move in .x16 groups: four pairs = 64 bytes per lane.
  TRPL_FN void st4(int p, const real* v) const {
    asm volatile("{\n .reg .b32 t0,t1,t2,t3,t4,t5,t6,t7;\n mov.b64 {t0,t1}, %1;\n mov.b64 {t2,t3}, %2;\n"
                 " mov.b64 {t4,t5}, %3;\n mov.b64 {t6,t7}, %4;\n"
                 " tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {t0,t1,t2,t3,t4,t5,t6,t7};\n}"
                 :: "r"(base + 4u * (unsigned)p), "d"(v[0]), "d"(v[1]), "d"(v[2]), "d"(v[3]) : "memory");
  }
  TRPL_FN void ld4(int p, real* v) const {
    asm volatile("{\n .reg .b32 t0,t1,t2,t3,t4,t5,t6,t7;\n"
                 " tcgen05.ld.sync.aligned.32x32b.x8.b32 {t0,t1,t2,t3,t4,t5,t6,t7}, [%4];\n"
                 " mov.b64 %0, {t0,t1};\n mov.b64 %1, {t2,t3};\n mov.b64 %2, {t4,t5};\n mov.b64 %3, {t6,t7};\n}"
                 : "=d"(v[0]), "=d"(v[1]), "=d"(v[2]), "=d"(v[3]) : "r"(base + 4u * (unsigned)p) : "memory");
  }
  TRPL_FN void st8(int p, const real* v) const {
    asm volatile("{\n .reg .b32 t<16>;\n mov.b64 {t0,t1}, %1;\n mov.b64 {t2,t3}, %2;\n mov.b64 {t4,t5}, %3;\n"
                 " mov.b64 {t6,t7}, %4;\n mov.b64 {t8,t9}, %5;\n mov.b64 {t10,t11}, %6;\n mov.b64 {t12,t13}, %7;\n"
                 " mov.b64 {t14,t15}, %8;\n"
                 " tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {t0,t1,t2,t3,t4,t5,t6,t7,t8,t9,t10,t11,t12,t13,t14,t15};\n}"
                 :: "r"(base + 4u * (unsigned)p), "d"(v[0]), "d"(v[1]), "d"(v[2]), "d"(v[3]), "d"(v[4]), "d"(v[5]),
                    "d"(v[6]), "d"(v[7]) : "memory");
  }
  TRPL_FN void ld8(int p, real* v) const {
    asm volatile("{\n .reg .b32 t<16>;\n"
                 " tcgen05.ld.sync.aligned.32x32b.x16.b32 {t0,t1,t2,t3,t4,t5,t6,t7,t8,t9,t10,t11,t12,t13,t14,t15}, [%8];\n"
                 " mov.b64 %0, {t0,t1};\n mov.b64 %1, {t2,t3};\n mov.b64 %2, {t4,t5};\n mov.b64 %3, {t6,t7};\n"
                 " mov.b64 %4, {t8,t9};\n mov.b64 %5, {t10,t11};\n mov.b64 %6, {t12,t13};\n mov.b64 %7, {t14,t15};\n}"
                 : "=d"(v[0]), "=d"(v[1]), "=d"(v[2]), "=d"(v[3]), "=d"(v[4]), "=d"(v[5]), "=d"(v[6]), "=d"(v[7])
                 : "r"(base + 4u * (unsigned)p) : "memory");
  }
  TRPL_FN void wait_ld() const { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
  TRPL_FN void wait_st() const { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
};
// the same interface on shared memory, so that a region can live in either
TRPL_FN void mem_wait_ld(const LaneMem&) {}
TRPL_FN void mem_wait_st(const LaneMem&) {}
TRPL_FN void mem_wait_ld(const LaneTm& t) { t.wait_ld(); }
TRPL_FN void mem_wait_st(const LaneTm& t) { t.wait_st(); }
// N consecutive pairs <-> 2N values, in the widest moves the memory has
template <int N> TRPL_FN void mem_ld_pairs(const LaneMem& m, int p, real* v) {
  TRPL_UNROLL for (int i = 0; i < N; ++i) m.ld2(p + i, v[2 * i], v[2 * i + 1]);
}
template <int N> TRPL_FN void mem_st_pairs(const LaneMem& m, int p, const real* v) {
  TRPL_UNROLL for (int i = 0; i < N; ++i) m.st2(p + i, v[2 * i], v[2 * i + 1]);
}
template <int N> TRPL_FN void mem_ld_pairs(const LaneTm& m, int p, real* v) {
  constexpr int G = N / 4;
  TRPL_UNROLL for (int g = 0; g < G; ++g) m.ld8(p + 4 * g, v + 8 * g);
  if constexpr ((N & 3) >= 2) m.ld4(p + 4 * G, v + 8 * G);
  if constexpr (N & 1) m.ld2(p + N - 1, v[2 * N - 2], v[2 * N - 1]);
}
template <int N> TRPL_FN void mem_st_pairs(const LaneTm& m, int p, const real* v) {
  constexpr int G = N / 4;
  TRPL_UNROLL for (int g = 0; g < G; ++g) m.st8(p + 4 * g, v + 8 * g);
  if constexpr ((N & 3) >= 2) m.st4(p + 4 * G, v + 8 * G);
  if constexpr (N & 1) m.st2(p + N - 1, v[2 * N - 2], v[2 * N - 1]);
}
}  // namespace simt

#else
// ------------------------------------------------------------------------------------------
// host lock-step emulation (tests only)
// ------------------------------------------------------------------------------------------
#include <vector>
#include <algorithm>
#include <stdio.h>
#include <stdlib.h>
#define TRPL_FN inline
#define TRPL_HD inline
#define TRPL_UNROLL
#define TRPL_UNROLL4

namespace simt {
constexpr int LANES = 32 * TRPL_TEAM;
constexpr int LOG2_LANES = TRPL_TEAM == 4 ? 7 : TRPL_TEAM == 2 ? 6 : 5;
#if TRPL_TEAM == 4
typedef unsigned __int128 lanebits;
#else
typedef unsigned long long lanebits;
#endif
struct real {
  double v[LANES];
  real() {}
  real(double x) { for (int i = 0; i < LANES; ++i) v[i] = x; }
};
struct mask { bool v[LANES]; };
struct ivec { int v[LANES]; };

#define TRPL_BIN(op)                                                                          \
  inline real operator op(const real& a, const real& b) { real r; for (int i = 0; i < LANES; ++i) r.v[i] = a.v[i] op b.v[i]; return r; } \
  inline real operator op(const real& a, double b) { real r; for (int i = 0; i < LANES; ++i) r.v[i] = a.v[i] op b; return r; }           \
  inline real operator op(double a, const real& b) { real r; for (int i = 0; i < LANES; ++i) r.v[i] = a op b.v[i]; return r; }
TRPL_BIN(+) TRPL_BIN(-) TRPL_BIN(*) TRPL_BIN(/)
#undef TRPL_BIN
inline real operator-(const real& a) { real r; for (int i = 0; i < LANES; ++i) r.v[i] = -a.v[i]; return r; }
inline real& operator+=(real& a, const real& b) { for (int i = 0; i < LANES; ++i) a.v[i] += b.v[i]; return a; }
inline real& operator-=(real& a, const real& b) { for (int i = 0; i < LANES; ++i) a.v[i] -= b.v[i]; return a; }
inline real& operator*=(real& a, const real& b) { for (int i = 0; i < LANES; ++i) a.v[i] *= b.v[i]; return a; }
#define TRPL_CMP(op)                                                                          \
  inline mask operator op(const real& a, const real& b) { mask r; for (int i = 0; i < LANES; ++i) r.v[i] = a.v[i] op b.v[i]; return r; } \
  inline mask operator op(const real& a, double b) { mask r; for (int i = 0; i < LANES; ++i) r.v[i] = a.v[i] op b; return r; }
TRPL_CMP(<) TRPL_CMP(<=) TRPL_CMP(>) TRPL_CMP(>=) TRPL_CMP(!=) TRPL_CMP(==)
#undef TRPL_CMP
#define TRPL_ICMP(op)                                                                         \
  inline mask operator op(const ivec& a, int b) { mask r; for (int i = 0; i < LANES; ++i) r.v[i] = a.v[i] op b; return r; } \
  inline mask operator op(const ivec& a, const ivec& b) { mask r; for (int i = 0; i < LANES; ++i) r.v[i] = a.v[i] op b.v[i]; return r; }
TRPL_ICMP(<) TRPL_ICMP(<=) TRPL_ICMP(>) TRPL_ICMP(>=) TRPL_ICMP(==) TRPL_ICMP(!=)
#undef TRPL_ICMP

inline ivec lane_id() { ivec r; for (int i = 0; i < LANES; ++i) r.v[i] = i; return r; }
inline real splat(double x) { return real(x); }
inline double uni(const real& x) { return x.v[0]; }
inline double lane0(const real& x) { return x.v[0]; }
inline real shfl_up(const real& x, int d) { real r; for (int i = 0; i < LANES; ++i) r.v[i] = (i - d >= 0) ? x.v[i - d] : x.v[i]; return r; }
inline real shfl_down(const real& x, int d) { real r; for (int i = 0; i < LANES; ++i) r.v[i] = (i + d < LANES) ? x.v[i + d] : x.v[i]; return r; }
inline real shfl_idx(const real& x, int s) { return real(x.v[s]); }
template <int N> inline void nbr_up(const real (&x)[N], real (&y)[N]) { for (int i = 0; i < N; ++i) y[i] = shfl_up(x[i], 1); }
template <int N> inline void nbr_down(const real (&x)[N], real (&y)[N]) { for (int i = 0; i < N; ++i) y[i] = shfl_down(x[i], 1); }
template <int NU, int ND> inline void nbr_both(const real (&xu)[NU], real (&yu)[NU], const real (&xd)[ND], real (&yd)[ND]) {
  nbr_up<NU>(xu, yu); nbr_down<ND>(xd, yd);
}
inline real sel3(const mask& m, const real& a, const real& b) { real r; for (int i = 0; i < LANES; ++i) r.v[i] = m.v[i] ? a.v[i] : b.v[i]; return r; }
template <class A, class B> inline real sel(const mask& m, const A& a, const B& b) { return sel3(m, real(a), real(b)); }
inline ivec seli(const mask& m, const ivec& a, const ivec& b) { ivec r; for (int i = 0; i < LANES; ++i) r.v[i] = m.v[i] ? a.v[i] : b.v[i]; return r; }
inline mask mand(const mask& a, const mask& b) { mask r; for (int i = 0; i < LANES; ++i) r.v[i] = a.v[i] && b.v[i]; return r; }
inline mask mor(const mask& a, const mask& b) { mask r; for (int i = 0; i < LANES; ++i) r.v[i] = a.v[i] || b.v[i]; return r; }
inline mask mnot(const mask& a) { mask r; for (int i = 0; i < LANES; ++i) r.v[i] = !a.v[i]; return r; }
inline mask mconst(bool b) { mask r; for (int i = 0; i < LANES; ++i) r.v[i] = b; return r; }
inline bool warp_any(const mask& m) { for (int i = 0; i < LANES; ++i) if (m.v[i]) return true; return false; }
inline lanebits warp_ballot(const mask& m) { lanebits b = 0; for (int i = 0; i < LANES; ++i) if (m.v[i]) b |= ((lanebits)1 << i); return b; }
inline mask lane_lt(const ivec& l, int k) { return l < k; }
inline bool local_any(const mask& m) { for (int i = 0; i < LANES; ++i) if (m.v[i]) return true; return false; }
inline real fmadd3(const real& a, const real& b, const real& c) { real r; for (int i = 0; i < LANES; ++i) r.v[i] = fma(a.v[i], b.v[i], c.v[i]); return r; }
template <class A, class B, class C> inline real fmadd(const A& a, const B& b, const C& c) { return fmadd3(real(a), real(b), real(c)); }
inline real vdiv(const real& a, const real& b) { return a / b; }
inline real rcp_approx(const real& x) { real r; for (int i = 0; i < LANES; ++i) r.v[i] = 1.0 / x.v[i]; return r; }
inline real vmax_fast(const real& a, const real& b) { real r; for (int i = 0; i < LANES; ++i) r.v[i] = a.v[i] > b.v[i] ? a.v[i] : b.v[i]; return r; }
inline float ctl_powf(float x, float y) { return powf(x, y); }
inline real rcp(const real& x) { real r; for (int i = 0; i < LANES; ++i) r.v[i] = 1.0 / x.v[i]; return r; }
#define TRPL_UN(name, expr) inline real name(const real& x) { real r; for (int i = 0; i < LANES; ++i) { double a = x.v[i]; r.v[i] = (expr); } return r; }
TRPL_UN(vabs, fabs(a)) TRPL_UN(vexp, exp(a)) TRPL_UN(vlog, log(a)) TRPL_UN(vlog10, log10(a)) TRPL_UN(vsqrt, sqrt(a))
#undef TRPL_UN
inline real vmax2(const real& a, const real& b) { real r; for (int i = 0; i < LANES; ++i) r.v[i] = fmax(a.v[i], b.v[i]); return r; }
inline real vmin2(const real& a, const real& b) { real r; for (int i = 0; i < LANES; ++i) r.v[i] = fmin(a.v[i], b.v[i]); return r; }
template <class A, class B> inline real vmax(const A& a, const B& b) { return vmax2(real(a), real(b)); }
template <class A, class B> inline real vmin(const A& a, const B& b) { return vmin2(real(a), real(b)); }
inline mask is_nan(const real& x) { mask r; for (int i = 0; i < LANES; ++i) r.v[i] = (x.v[i] != x.v[i]); return r; }
inline real warp_sum(real x) {
  for (int o = 16; o > 0; o >>= 1) { real y; for (int i = 0; i < LANES; ++i) y.v[i] = x.v[i] + x.v[i ^ o]; x = y; }
  // several warps: the device build's order - each warp's partial, then (p0 + p1) [+ (p2 + p3)]
#if TRPL_TEAM == 2
  return real(x.v[0] + x.v[32]);
#elif TRPL_TEAM == 4
  return real((x.v[0] + x.v[32]) + (x.v[64] + x.v[96]));
#else
  return x;
#endif
}
inline real warp_max(real x) {
  for (int o = LANES / 2; o > 0; o >>= 1) { real y; for (int i = 0; i < LANES; ++i) y.v[i] = fmax(x.v[i], x.v[i ^ o]); x = y; }
  return x;
}
inline real warp_min(const real& x) { return -warp_max(-x); }
inline void warp_sum2(real& a, real& b) { a = warp_sum(a); b = warp_sum(b); }
inline real warp_scan_incl(real x) {
  // (two warps: a scan inside each warp, then the first warp's total onto the second, as on the device)
  for (int o = 1; o < 32; o <<= 1) { real y = x; for (int i = 0; i < LANES; ++i) if ((i & 31) >= o) y.v[i] = x.v[i] + x.v[i - o]; x = y; }
  if (LANES > 32) {
    double tot[LANES / 32];
    for (int w = 0; w < LANES / 32; ++w) tot[w] = x.v[32 * w + 31];
    for (int w = 1; w < LANES / 32; ++w) {
      double off = tot[0];
      for (int k = 1; k < w; ++k) off = off + tot[k];
      for (int i = 32 * w; i < 32 * w + 32; ++i) x.v[i] += off;
    }
  }
  return x;
}
inline real gather(const double* p, const ivec& idx, const mask& m, double other) {
  real r; for (int i = 0; i < LANES; ++i) r.v[i] = m.v[i] ? p[idx.v[i]] : other; return r;
}
inline void gather2(const double* p, const ivec& idx, const mask& m, double other, real& a, real& b) {
  for (int i = 0; i < LANES; ++i) { a.v[i] = m.v[i] ? p[idx.v[i]] : other; b.v[i] = m.v[i] ? p[idx.v[i] + 1] : other; }
}
inline void scatter(double* p, const ivec& idx, const mask& m, const real& v) {
  for (int i = 0; i < LANES; ++i) if (m.v[i]) p[idx.v[i]] = v.v[i];
}
inline ivec iadd(const ivec& a, int b) { ivec r; for (int i = 0; i < LANES; ++i) r.v[i] = a.v[i] + b; return r; }
inline ivec imul(const ivec& a, int b) { ivec r; for (int i = 0; i < LANES; ++i) r.v[i] = a.v[i] * b; return r; }
inline ivec iaddv(const ivec& a, const ivec& b) { ivec r; for (int i = 0; i < LANES; ++i) r.v[i] = a.v[i] + b.v[i]; return r; }
inline ivec isubv(const ivec& a, const ivec& b) { ivec r; for (int i = 0; i < LANES; ++i) r.v[i] = a.v[i] - b.v[i]; return r; }
inline ivec ishr1(const ivec& a) { ivec r; for (int i = 0; i < LANES; ++i) r.v[i] = a.v[i] >> 1; return r; }
inline ivec iclamp(const ivec& a, int lo, int hi) { ivec r; for (int i = 0; i < LANES; ++i) r.v[i] = a.v[i] < lo ? lo : (a.v[i] > hi ? hi : a.v[i]); return r; }
inline ivec isplat(int a) { ivec r; for (int i = 0; i < LANES; ++i) r.v[i] = a; return r; }
inline ivec irsub(int a, const ivec& b) { ivec r; for (int i = 0; i < LANES; ++i) r.v[i] = a - b.v[i]; return r; }
inline ivec lane_minus(int d) { ivec r; for (int i = 0; i < LANES; ++i) r.v[i] = i >= d ? i - d : i; return r; }
inline ivec lane_plus(int d) { ivec r; for (int i = 0; i < LANES; ++i) r.v[i] = i + d < LANES ? i + d : i; return r; }
inline ivec to_int_floor(const real& x) { ivec r; for (int i = 0; i < LANES; ++i) r.v[i] = (int)floor(x.v[i]); return r; }
inline real to_real(const ivec& a) { real r; for (int i = 0; i < LANES; ++i) r.v[i] = (double)a.v[i]; return r; }

// every access is bounds-checked (std::vector::at): the pair indices are the same compile-time
// layout constants the device build uses, so the CPU test tier doubles as the bounds check of the
// shared-memory and tensor-memory slices (compute-sanitizer is not available on the GPU pool)
struct LaneMem {
  std::vector<real> slots;     // 2 per pair
  explicit LaneMem(int n_pairs) : slots(2 * n_pairs) {}
  void ld2(int p, real& a, real& b) const { a = slots.at(2 * p); b = slots.at(2 * p + 1); }
  void st2(int p, const real& a, const real& b) { slots.at(2 * p) = a; slots.at(2 * p + 1) = b; }
  void ld2_from(int p, const ivec& src, real& a, real& b) const {
    for (int i = 0; i < LANES; ++i) { a.v[i] = slots.at(2 * p).v[src.v[i] & (LANES - 1)]; b.v[i] = slots.at(2 * p + 1).v[src.v[i] & (LANES - 1)]; }
  }
  double uld(int p, int i) const { return slots.at(2 * p + (i & 1)).v[i >> 1]; }
  void ust(int p, int i, double v) { slots.at(2 * p + (i & 1)).v[i >> 1] = v; }
};
#if TRPL_TEAM >= 2
inline void team_other_sync();
inline void warp_sync() { team_other_sync(); }
#else
inline void warp_sync() {}
#endif
// host stand-in of the tensor-memory slice (see the device half): just another array of pairs
struct LaneTm {
  std::vector<real> slots;
  explicit LaneTm(int n_pairs) : slots(2 * n_pairs) {}
  void ld2(int p, real& a, real& b) const { a = slots.at(2 * p); b = slots.at(2 * p + 1); }
  void st2(int p, const real& a, const real& b) { slots.at(2 * p) = a; slots.at(2 * p + 1) = b; }
};
template <class M> inline void mem_wait_ld(const M&) {}
template <class M> inline void mem_wait_st(const M&) {}
template <int N, class M> inline void mem_ld_pairs(const M& m, int p, real* v) { for (int i = 0; i < N; ++i) m.ld2(p + i, v[2 * i], v[2 * i + 1]); }
template <int N, class M> inline void mem_st_pairs(M& m, int p, const real* v) { for (int i = 0; i < N; ++i) m.st2(p + i, v[2 * i], v[2 * i + 1]); }
#if TRPL_TEAM >= 2
// The device build's mailbox discipline, checked: two consecutive team primitives of a trajectory
// must not use the same mailbox slot (see the device half).  Slot numbers come from the same macros.
inline int& team_last_slot() { static thread_local int last = -1; return last; }
inline void team_slot_check(int s) {
  if (team_last_slot() == s) { fprintf(stderr, "simt: mailbox slot %d used by two consecutive team primitives\n", s); abort(); }
  team_last_slot() = s;
}
inline void team_other_sync() { team_last_slot() = -1; }     // a barrier that uses no mailbox (warp_sync)
template <int S> inline double lane0_s(const real& x) { team_slot_check(S); return lane0(x); }
template <int S> inline real shfl_idx_s(const real& x, int s) { team_slot_check(S); return shfl_idx(x, s); }
template <int S> inline real shfl_up_s(const real& x, int d) { team_slot_check(S); if (d != 1) abort(); return shfl_up(x, d); }
template <int S> inline real shfl_down_s(const real& x, int d) { team_slot_check(S); if (d != 1) abort(); return shfl_down(x, d); }
template <int S> inline bool warp_any_s(const mask& m) { team_slot_check(S); return warp_any(m); }
template <int S> inline lanebits warp_ballot_s(const mask& m) { team_slot_check(S); return warp_ballot(m); }
template <int S> inline real warp_sum_s(const real& x) { team_slot_check(S); return warp_sum(x); }
template <int S> inline real warp_max_s(const real& x) { team_slot_check(S); return warp_max(x); }
template <int S> inline real warp_min_s(const real& x) { team_slot_check(S); return warp_min(x); }
template <int S> inline real warp_scan_incl_s(const real& x) { team_slot_check(S); return warp_scan_incl(x); }
template <int S> inline void warp_sum2_s(real& a, real& b) { team_slot_check(S); warp_sum2(a, b); }
template <int S, int N> inline void nbr_up_s(const real (&x)[N], real (&y)[N]) { team_slot_check(S); nbr_up<N>(x, y); }
template <int S, int N> inline void nbr_down_s(const real (&x)[N], real (&y)[N]) { team_slot_check(S); nbr_down<N>(x, y); }
template <int S, int NU, int ND> inline void nbr_both_s(const real (&xu)[NU], real (&yu)[NU], const real (&xd)[ND], real (&yd)[ND]) {
  team_slot_check(S); nbr_both<NU, ND>(xu, yu, xd, yd);
}
#endif
}  // namespace simt
#endif

#if TRPL_TEAM >= 2
// One mailbox slot per call site (see the device half of the team vocabulary).
#define TRPL_TEAM_SLOT (__COUNTER__ & 63)
#define lane0(x) lane0_s<TRPL_TEAM_SLOT>(x)
#define shfl_idx(x, s) shfl_idx_s<TRPL_TEAM_SLOT>(x, s)
#define shfl_up(x, d) shfl_up_s<TRPL_TEAM_SLOT>(x, d)
#define shfl_down(x, d) shfl_down_s<TRPL_TEAM_SLOT>(x, d)
#define warp_any(m) warp_any_s<TRPL_TEAM_SLOT>(m)
#define warp_ballot(m) warp_ballot_s<TRPL_TEAM_SLOT>(m)
#define warp_sum(x) warp_sum_s<TRPL_TEAM_SLOT>(x)
#define warp_max(x) warp_max_s<TRPL_TEAM_SLOT>(x)
#define warp_min(x) warp_min_s<TRPL_TEAM_SLOT>(x)
#define warp_scan_incl(x) warp_scan_incl_s<TRPL_TEAM_SLOT>(x)
#define warp_sum2 warp_sum2_s<TRPL_TEAM_SLOT>
#define nbr_up nbr_up_s<TRPL_TEAM_SLOT>
#define nbr_down nbr_down_s<TRPL_TEAM_SLOT>
#define nbr_both nbr_both_s<TRPL_TEAM_SLOT>
#endif
