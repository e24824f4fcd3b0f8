// trajectory.h - one (parameter set, measurement) trajectory, start to finish, inside one warp:
// initial condition -> adaptive RODAS4 time integration -> PL/TRTS readout at the measurement
// times -> log-likelihood against the measurement.  Replaces, for one trajectory,
//   forward_solver.py:41-203   solve()            (init, LSODA integration, PL readout, min_y floor)
//   trial_move_evaluation.py:96-166 one_sim_likelihood() (abs/negative test, log10 residual, sum)
//
// Integrator: RODAS4 (Hairer & Wanner, Solving ODEs II, sec. IV.7/IV.10; 6 stages, order 4(3),
// stiffly accurate, L-stable, gamma = 1/4), exact Jacobian every step, error = 6th stage.
// The coefficient set is verified against the order conditions in tools/proto/check_rodas_coeffs.py.
// Step control: Gustafsson predictive controller, all norms reduced with warp shuffles.
// Output: quintic Hermite interpolation of ln(signal) through the last three step points
// (value + time derivative, both by warp reductions), evaluated by the lanes in parallel.
#pragma once
#include <float.h>
#include "simt.h"
#include "model.h"
#include "blocktri.h"
#include "irf.h"

namespace trpl {
using namespace simt;

#if defined(TRPL_FN) && defined(__CUDACC__) && !defined(TRPL_HOST_EMU)
#define TRPL_CONST __constant__ const
#define TRPL_NOINLINE __device__ __noinline__
#else
#define TRPL_CONST static const
#define TRPL_NOINLINE static
#endif

// RODAS4 in the Hairer-Wanner "transformed" form:
//   (1/(gamma h) I - J) K_i = f(u + sum_j a_ij K_j) + sum_j (c_ij / h) K_j ,  u_new = u + sum m_i K_i
struct Rodas4 {
  static constexpr double A[6][6] = {
      {0, 0, 0, 0, 0, 0},
      {0.1544000000000000e+01, 0, 0, 0, 0, 0},
      {0.9466785280815826e+00, 0.2557011698983284e+00, 0, 0, 0, 0},
      {0.3314825187068521e+01, 0.2896124015972201e+01, 0.9986419139977817e+00, 0, 0, 0},
      {0.1221224509226641e+01, 0.6019134481288629e+01, 0.1253708332932087e+02, -0.6878860361058950e+00, 0, 0},
      {0.1221224509226641e+01, 0.6019134481288629e+01, 0.1253708332932087e+02, -0.6878860361058950e+00, 1.0, 0}};
  static constexpr double C[6][6] = {
      {0, 0, 0, 0, 0, 0},
      {-0.5668800000000000e+01, 0, 0, 0, 0, 0},
      {-0.2430093356833875e+01, -0.2063599157091915e+00, 0, 0, 0, 0},
      {-0.1073529058151375e+00, -0.9594562251023355e+01, -0.2047028614809616e+02, 0, 0, 0},
      {0.7496443313967647e+01, -0.1024680431464352e+02, -0.3399990352819905e+02, 0.1170890893206160e+02, 0, 0},
      {0.8083246795921522e+01, -0.7981132988064893e+01, -0.3152159432874371e+02, 0.1631930543123136e+02,
       -0.6058818238834054e+01, 0}};
};
constexpr double RODAS4_GAMMA = 0.25;

// Weight of the running-charge components in the error norm (see DESIGN.md section 2,
// "Tolerances"): Q is slaved to the densities by dielectric relaxation (sub-picosecond), the
// stiffly accurate integrator resolves it like an algebraic variable, and the embedded estimate
// for such components is known to be pessimistic.
// Tuning switches of the storage layout (measured on B200, DESIGN.md section 5)
#ifndef TRPL_PM_REGS
#define TRPL_PM_REGS 0            // PCR multipliers in registers (1) or in tensor/shared memory (0)
#endif
#ifndef TRPL_Q_ERR_WEIGHT
#define TRPL_Q_ERR_WEIGHT 0.03
#endif
constexpr double Q_ERR_WEIGHT = TRPL_Q_ERR_WEIGHT;
// The density error is controlled relative to the excess carrier density down to EXCESS_RANGE
// times its initial peak (12 decades of dynamic range; below that the scale stays at the floor).
#ifndef TRPL_EXCESS_RANGE
#define TRPL_EXCESS_RANGE 1e-12
#endif
constexpr double EXCESS_RANGE = TRPL_EXCESS_RANGE;
// safety factor of the step-size controller (Hairer's RODAS code uses 0.9; with the predictive controller rejections stay below 1% at 0.95)
#ifndef TRPL_CTL_SAFETY
#define TRPL_CTL_SAFETY 0.95f
#endif
constexpr float CTL_SAFETY = TRPL_CTL_SAFETY;

enum StatusBits {
  ST_OK = 0,
  ST_MAX_STEPS = 1,     // step budget exhausted before the last measurement time
  ST_H_UNDERFLOW = 2,   // step size collapsed
  ST_NONFINITE = 4,     // NaN/Inf state
  ST_FLOORED = 8,       // signal fell below DBL_MIN and was floored (forward_solver.py:190-192)
  ST_NEG_FRAC = 16,     // too many negative values (trial_move_evaluation.py:117-123) -> -inf
  ST_NAN_LL = 32,       // likelihood was NaN -> -inf (trial_move_evaluation.py:159-165)
  ST_CONV_FAIL = 64,    // IRF convolution failed -> -inf (trial_move_evaluation.py:83-87, :103-106)
  ST_EXPLICIT = 128     // informational: integrated by the explicit Runge-Kutta path (explicit.h)
};

enum OptFlags { OPT_FORCE_MIN_Y = 1, OPT_NO_LIKELIHOOD = 2, OPT_LADDER = 4, OPT_NO_EXPLICIT = 8, OPT_CTA_PER_TRAJ = 16,
                OPT_EXTRAPOLATION = 32, OPT_FIT = 64 };

struct SolverOpts {
  double rtol, atol;
  double hmax;          // <= 0: steps limited by the error controller only
  int max_steps;
  int flags;
};

// one measurement (shared by every parameter set)
struct MeasDesc {
  double thickness;
  double ini_a, ini_b;   // fluence mode: fluence [cm^-2], absorption [cm^-1]
  int nx;
  int meas_type;         // MeasType
  int ini_mode;          // 0 density profile, 1 fluence/absorption/direction
  int ini_dir;           // fluence mode: <0 reverses the profile
  int n_t;               // number of measurement times (times[0] == 0)
  int t_off;             // offset of this measurement in times/vals/uncs
  int prof_off;          // offset of this measurement's profile (density mode)
  int irf_nk;            // rows of this measurement's IRF moment table, 0 = no convolution
  double irf_dt;         // mean IRF time step [ns]
  int irf_off;           // first row of the table in the moments array
  int pad_;
  double min_y;          // floor of the simulated signal (Grid.min_y, sim_utils.py:281)
};

struct TrajIn {
  const double* par;     // TRPL_NPARAM model-unit parameters
  const MeasDesc* md;
  const double* times;   // [n_t]
  const double* vals;    // [n_t] log10 measurement (may be null with OPT_NO_LIKELIHOOD)
  const double* uncs;    // [n_t]
  const double* profile; // [nx] cm^-3 (density mode)
  double scale_shift;    // log10 of the curve's scale factor
  double s2T[3];         // model_uncertainty^2 * T for up to three temperatures
  double fl_mult, al_mult;
  double* curve;         // optional [n_t] simulated signal in measurement units
  bool post_pass;        // likelihood is taken in finalize_trajectory (min_y floor, IRF, ladder)
  double* hist;          // per-warp scratch: (t, S, dS/dt) of accepted steps, HIST_CAP entries
};

constexpr int HIST_CAP = 1024;

// Everything only the final pass needs.  Built AFTER the integration loop so that none of it is
// live (and spilled) across the hot loop.
struct TailIn {
  IrfDesc irf;           // irf.nk == 0: no convolution
  // tempering ladder (OPT_LADDER): likelihood at every ladder temperature; s2T[1] holds sigma^2
  const double* ladder_T;
  int ladder_n;
  double* ladder_out;    // [ladder_n]
  double* r2_scratch;    // [n_t] per-warp
  double* u2_scratch;    // [n_t] per-warp
};

// what the integration loop hands to the final pass
struct TrajMid {
  double l[3];           // streaming likelihood sums (valid when !post_pass)
  double n_neg;
};

struct TrajOut {
  double logll[3];
  int status, n_acc, n_rej;
};

// Storage of one trajectory besides its registers, in PAIRS (16 bytes per lane).  Two memories:
//   sm  the warp's slice of shared memory: whatever lanes exchange (PCR rows) or share (Coef)
//   tm  the warp's slice of tensor memory (simt.h LaneTm): lane-private data only - the stage
//       increments K_1..K_5, the interior factors / spikes / interface blocks, the trap
//       condensation coefficients.  These are 85% of the on-chip traffic of a step; on the
//       shared-memory pipe they made the kernel bandwidth-bound (DESIGN.md section 5).
// A CTA of four warps allocates TM_COLS columns; with at most 256 two CTAs share an SM's 512.
// Regions that do not fit the tensor-memory budget stay in shared memory.
template <int NPL, int MODEL>
struct Slots {
  static constexpr int NKS = 5;                                // stages kept (the 6th is consumed in registers)
  static constexpr int TPAIRS = (MODEL == MODEL_TRAPS) ? (NPL + 1) / 2 : 0;   // trap component, two nodes per pair
  static constexpr int KSTRIDE = NPL + TPAIRS;                 // pairs per stage: (K_N, K_Q) per node [+ K_T]
  static constexpr int KP = NKS * KSTRIDE;
  static constexpr int FACP = FacSlots<NPL>::COUNT;
  static constexpr int TRP = (MODEL == MODEL_TRAPS) ? 3 * NPL : 0;   // traps: 5 condensation coefficients per node
  // PCR multipliers: one level per doubling of the stride (5 for a warp, 6 for a two-warp team) x 4
  // pairs + the inverse (2 pairs, padded to 4)
  static constexpr int PMP = 4 * LOG2_LANES + 4;
#if TRPL_PM_REGS
  static constexpr bool PM_IN_REGS = true;
#else
  static constexpr bool PM_IN_REGS = false;
#endif
  // tensor-memory budget in pairs per warp: 512 columns / 2 CTAs per SM / 4 columns per pair
#ifdef TRPL_NO_TMEM
  static constexpr int TM_WANT = 0;
#else
  static constexpr int TM_WANT = 64;
#endif
  // one CTA per SM (128 pairs) for the grids whose factor blocks alone exceed the two-CTA budget (8
  // nodes per lane: no product kernel since the two-warp teams of team_kernels.cu, host lock-step
  // instantiation of the generic extrapolation driver only)
  static constexpr int TM_BUDGET = (TM_WANT == 64 && FACP > 64) ? 128 : TM_WANT;
  // priority: factor blocks, then multipliers (whole levels; the rest stays in shared memory),
  // then stage increments, then the trap coefficients
  static constexpr bool FAC_IN_TM = FACP <= TM_BUDGET;
  static constexpr int TM_LEFT1 = TM_BUDGET - (FAC_IN_TM ? FACP : 0);
  static constexpr int PM_TM_PAIRS = PM_IN_REGS ? 0 : (TM_LEFT1 >= PMP ? PMP : (TM_LEFT1 / 4) * 4);
  static constexpr int PM_SM_PAIRS = PM_IN_REGS ? 0 : (PM_TM_PAIRS == PMP ? 0 : PMP - 2 - PM_TM_PAIRS);
  static constexpr int TM_LEFT2 = TM_LEFT1 - PM_TM_PAIRS;
  static constexpr bool K_IN_TM = FAC_IN_TM && KP <= TM_LEFT2;
  static constexpr int TM_LEFT3 = TM_LEFT2 - (K_IN_TM ? KP : 0);
  static constexpr bool TRAP_IN_TM = K_IN_TM && TRP > 0 && TRP <= TM_LEFT3;
  // tensor memory: K | FAC | TRAP | PM | first increments   (K first: the explicit path runs its 7
  // stages from there)
  static constexpr int TM_K = 0;
  static constexpr int TM_FAC = K_IN_TM ? (KP + 3) / 4 * 4 : 0;
  static constexpr int TM_TRAP = TM_FAC + (FAC_IN_TM ? FACP : 0);
  static constexpr int TM_PM = (TM_TRAP + (TRAP_IN_TM ? TRP : 0) + 3) / 4 * 4;
  // When the increments as a whole stay in shared memory, whatever tensor memory is left takes the
  // first K_TM_STAGES of them: K_1 is read back by four later stages, K_2 by three, K_5 by none.
  static constexpr int TM_KS = (TM_PM + PM_TM_PAIRS + 3) / 4 * 4;
  static constexpr int K_TM_ROOM = (!K_IN_TM && FAC_IN_TM && KSTRIDE % 4 == 0 && TM_BUDGET > TM_KS)
                                       ? (TM_BUDGET - TM_KS) / KSTRIDE : 0;
  static constexpr int K_TM_STAGES = K_TM_ROOM > NKS - 1 ? NKS - 1 : K_TM_ROOM;
  static constexpr int TM_COUNT = K_TM_STAGES > 0 ? TM_KS + K_TM_STAGES * KSTRIDE : TM_PM + PM_TM_PAIRS;
  static constexpr int TM_COLS = TM_COUNT == 0 ? 0 : (4 * TM_COUNT <= 32 ? 32 : 4 * TM_COUNT <= 64 ? 64 :
                                  4 * TM_COUNT <= 128 ? 128 : 4 * TM_COUNT <= 256 ? 256 : 512);
  // shared memory: [K] | [FAC] | [TRAP] | [PM rest] | XCH | UNI
  static constexpr int SM_K = 0;
  static constexpr int SM_FAC = K_IN_TM ? 0 : KP;
  static constexpr int SM_TRAP = SM_FAC + (FAC_IN_TM ? 0 : FACP);
  static constexpr int SM_PM = SM_TRAP + (TRAP_IN_TM ? 0 : TRP);
  // lane-exchange scratch: 2 pairs for the solves; the factorisation needs 12 (2 x 6, double
  // buffered) and borrows the K region when that lives in shared memory (dead at that point)
  static constexpr int XCH = SM_PM + PM_SM_PAIRS;
  static constexpr bool XCH_BORROWS_K = !K_IN_TM && KP >= 12;
  static constexpr int XCH_PAIRS = XCH_BORROWS_K ? 2 : 12;
  static constexpr int XCH_FACTOR = XCH_BORROWS_K ? SM_K : XCH;
  // one slot of warp-uniform scalars (Coef), behind everything else; when the increments live in
  // shared memory the slice is at least the 7 stages the explicit path keeps from KBASE on
  static constexpr int UNI = (K_IN_TM || XCH + XCH_PAIRS >= 7 * KSTRIDE) ? XCH + XCH_PAIRS : 7 * KSTRIDE;
  static constexpr int COUNT = UNI + 1;
  static constexpr int BYTES = COUNT * LANES * 16;
  // region bases in whichever memory holds them
  static constexpr int KBASE = K_IN_TM ? TM_K : SM_K;
  static constexpr int FAC = FAC_IN_TM ? TM_FAC : SM_FAC;
  static constexpr int TRAP = TRAP_IN_TM ? TM_TRAP : SM_TRAP;
  // contiguous pairs available from KBASE on (the explicit Runge-Kutta path keeps 7 stages there)
  static constexpr int KCAP = K_IN_TM ? TM_PM : UNI;
};

struct TrajMem {
  LaneMem sm;
  LaneTm tm;
};
// where the PCR multipliers live for this layout (blocktri.h PmRegs / PmRun)
template <class SL, bool REGS = SL::PM_IN_REGS>
struct PmChoice {
  typedef PmRegs type;
  TRPL_FN static type make(TrajMem&) { return type(); }
};
template <class SL>
struct PmChoice<SL, false> {
  typedef PmRun<LaneTm, LaneMem, SL::TM_PM, SL::SM_PM, SL::PM_TM_PAIRS> type;
  TRPL_FN static type make(TrajMem& m) { return type{m.tm, m.sm}; }
};
template <class SL> TRPL_FN auto& kmem(TrajMem& m) { if constexpr (SL::K_IN_TM) return m.tm; else return m.sm; }
template <class SL> TRPL_FN auto& fmem(TrajMem& m) { if constexpr (SL::FAC_IN_TM) return m.tm; else return m.sm; }
template <class SL> TRPL_FN auto& trmem(TrajMem& m) { if constexpr (SL::TRAP_IN_TM) return m.tm; else return m.sm; }

// stage increment K_s <-> its memory: one run of KSTRIDE pairs, (K_N, K_Q) per node [+ K_T two per pair]
template <int NPL, int MODEL, class M>
TRPL_FN void store_k(M& km, int kb, const Vec<NPL, MODEL>& k) {
  typedef Slots<NPL, MODEL> SL;
  real v[2 * SL::KSTRIDE];
  TRPL_UNROLL for (int j = 0; j < NPL; ++j) { v[2 * j] = k.n[j]; v[2 * j + 1] = k.q[j]; }
  if (MODEL == MODEL_TRAPS) {
    TRPL_UNROLL for (int j = 0; j < 2 * SL::TPAIRS; ++j) v[2 * NPL + j] = k.t[j < NPL ? j : NPL - 1];
  }
  mem_st_pairs<SL::KSTRIDE>(km, kb, v);
}
// issue the loads of one increment into a staging run (the caller waits, then unpacks)
template <int NPL, int MODEL>
struct KRun { real v[2 * Slots<NPL, MODEL>::KSTRIDE]; };
template <int NPL, int MODEL, class M>
TRPL_FN void load_k_nowait(const M& km, int kb, KRun<NPL, MODEL>& r) {
  mem_ld_pairs<Slots<NPL, MODEL>::KSTRIDE>(km, kb, r.v);
}
template <int NPL, int MODEL>
TRPL_FN void unpack_k(const KRun<NPL, MODEL>& r, Vec<NPL, MODEL>& k) {
  TRPL_UNROLL for (int j = 0; j < NPL; ++j) { k.n[j] = r.v[2 * j]; k.q[j] = r.v[2 * j + 1]; }
  if (MODEL == MODEL_TRAPS) {
    TRPL_UNROLL for (int j = 0; j < NPL; ++j) k.t[j] = r.v[2 * NPL + j];
  } else {
    k.t[0] = splat(0.0);
  }
}
// increment of stage `st` (0-based) of the Rosenbrock step: tensor memory for the first
// K_TM_STAGES stages when the K region is split, the K region's memory otherwise
template <int NPL, int MODEL>
TRPL_FN void store_stage(TrajMem& mem, int st, const Vec<NPL, MODEL>& k) {
  typedef Slots<NPL, MODEL> SL;
  if (SL::K_TM_STAGES > 0 && st < SL::K_TM_STAGES) store_k<NPL, MODEL>(mem.tm, SL::TM_KS + st * SL::KSTRIDE, k);
  else store_k<NPL, MODEL>(kmem<SL>(mem), SL::KBASE + st * SL::KSTRIDE, k);
}
template <int ST, int NPL, int MODEL>
TRPL_FN void load_stage_nowait(TrajMem& mem, KRun<NPL, MODEL>& r) {
  typedef Slots<NPL, MODEL> SL;
  if constexpr (ST < SL::K_TM_STAGES) load_k_nowait<NPL, MODEL>(mem.tm, SL::TM_KS + ST * SL::KSTRIDE, r);
  else load_k_nowait<NPL, MODEL>(kmem<SL>(mem), SL::KBASE + ST * SL::KSTRIDE, r);
}
template <int ST, int NPL, int MODEL>
TRPL_FN void wait_stage(TrajMem& mem) {
  typedef Slots<NPL, MODEL> SL;
  if constexpr (ST < SL::K_TM_STAGES) mem_wait_ld(mem.tm); else mem_wait_ld(kmem<SL>(mem));
}
template <int NPL, int MODEL>
TRPL_FN void fence_stage_stores(TrajMem& mem) {
  typedef Slots<NPL, MODEL> SL;
  if constexpr (SL::K_TM_STAGES > 0) mem_wait_st(mem.tm);
  mem_wait_st(kmem<SL>(mem));
}
template <int NPL, int MODEL, class M>
TRPL_FN void load_k(const M& km, int kb, Vec<NPL, MODEL>& k) {
  KRun<NPL, MODEL> r;
  mem_wait_st(km);
  load_k_nowait<NPL, MODEL>(km, kb, r);
  mem_wait_ld(km);
  unpack_k<NPL, MODEL>(r, k);
}

// ---- readout: signal and its time derivative, reduced over the warp --------------------------
template <int NPL, int MODEL>
TRPL_FN void readout(const Coef& c, const NodeMask<NPL>& m, int meas_type, const Vec<NPL, MODEL>& u,
                     const Vec<NPL, MODEL>& f, const RhsAux<NPL>& aux, double& val, double& dval) {
  real fql0 = shfl_up(f.q[NPL - 1], 1);
  fql0 = sel(m.first_lane, 0.0, fql0);
  real acc = splat(0.0), dacc = splat(0.0);
  TRPL_UNROLL for (int j = 0; j < NPL; ++j) {
    const real fql = (j == 0) ? fql0 : f.q[j - 1];
    real fp = f.n[j] + (f.q[j] - fql);
    if (MODEL == MODEL_TRAPS) fp = fp + f.t[j];
    real a, d;
    if (meas_type == MEAS_TRPL) {                       // forward_solver.py:228-236,267-269
      a = fmadd(u.n[j], aux.p[j], -c.n0p0);
      d = fmadd(f.n[j], aux.p[j], u.n[j] * fp);
    } else {                                            // forward_solver.py:239-247,272-274
      a = fmadd(c.mun, u.n[j] - c.n0, c.mup * (aux.p[j] - c.p0));
      d = fmadd(c.mun, f.n[j], c.mup * fp);
    }
    acc = acc + sel(m.real_node[j], a, 0.0);
    dacc = dacc + sel(m.real_node[j], d, 0.0);
  }
  const double scale = (meas_type == MEAS_TRPL) ? c.ks * c.dx * 1e23 : Q_COULOMB * c.dx * 1e9;
  warp_sum2(acc, dacc);
  val = uni(acc) * scale;
  dval = uni(dacc) * scale;
}

// ---- dense output: per-lane Hermite interpolation through logged step points -----------------
// Each lane interpolates its own measurement time.  Newton form on the doubled nodes
// [t1,t1,t2,t2,t0,t0] (t1,t2 = the step containing the time; t0 = the step point before it);
// `three` is false for the first step of a trajectory (cubic through two points).  Interpolation
// is done on ln(signal) whenever all points involved are positive.
TRPL_FN real hermite_lane(const real& tq, const mask& three, const real& t0, const real& y0, const real& s0,
                          const real& t1, const real& y1, const real& s1, const real& t2, const real& y2,
                          const real& s2) {
  const mask in_log = mand(mand(y1 > 0.0, y2 > 0.0), mor(mnot(three), y0 > 0.0));
  const mask log0 = mand(in_log, three);
  const real v1 = sel(in_log, vlog(sel(in_log, y1, 1.0)), y1);
  const real v2 = sel(in_log, vlog(sel(in_log, y2, 1.0)), y2);
  const real v0 = sel(in_log, sel(three, vlog(sel(log0, y0, 1.0)), 0.0), y0);
  const real d1 = sel(in_log, vdiv(s1, sel(in_log, y1, 1.0)), s1);
  const real d2 = sel(in_log, vdiv(s2, sel(in_log, y2, 1.0)), s2);
  const real d0 = sel(in_log, sel(three, vdiv(s0, sel(log0, y0, 1.0)), 0.0), s0);
  const real i21 = vdiv(splat(1.0), t2 - t1);
  const real f12 = (v2 - v1) * i21;
  const real f112 = (f12 - d1) * i21;
  const real f122 = (d2 - f12) * i21;
  const real f1122 = (f122 - f112) * i21;
  // the three-point part is garbage (and discarded) on lanes where `three` is false
  const real i01 = vdiv(splat(1.0), sel(three, t0 - t1, 1.0)), i02 = vdiv(splat(1.0), sel(three, t0 - t2, 1.0));
  const real f20 = (v0 - v2) * i02;
  const real f220 = (f20 - d2) * i02;
  const real f200 = (d0 - f20) * i02;
  const real f1220 = (f220 - f122) * i01;
  const real f2200 = (f200 - f220) * i02;
  const real f11220 = (f1220 - f1122) * i01;
  const real f12200 = (f2200 - f1220) * i01;
  const real c4 = sel(three, f11220, 0.0);
  const real c5 = sel(three, (f12200 - f11220) * i01, 0.0);
  const real a = tq - t1, b = tq - t2, e = tq - t0;
  const real a2 = a * a, b2 = b * b;
  real p = fmadd(e, c5, c4);                  // c4 + c5 (t-t0)
  p = fmadd(p, b2, fmadd(b, f1122, f112));    // c2 + c3 (t-t2) + (t-t2)^2 (...)
  p = fmadd(p, a2, fmadd(a, d1, v1));         // c0 + c1 (t-t1) + (t-t1)^2 (...)
  real y = sel(in_log, vexp(sel(in_log, p, 0.0)), p);
  // Guard: a smooth signal stays inside the band spanned by the step's two end values (plus one
  // span of margin).  When the signal has decayed into rounding noise the controller takes huge
  // steps and the high-order interpolant of noisy data can overshoot by tens of decades; those
  // points fall back to (log-)linear interpolation between the two ends.
  const real mn = vmin(y1, y2), mx = vmax(y1, y2);
  const real margin = (mx - mn) + 1e-6 * vabs(mx);
  const mask outside = mnot(mand(y >= mn - margin, y <= mx + margin));    // true for NaN
  if (warp_any(outside)) {
    const mask ends_log = mand(y1 > 0.0, y2 > 0.0);
    const real e1 = sel(ends_log, vlog(sel(ends_log, y1, 1.0)), y1);
    const real e2 = sel(ends_log, vlog(sel(ends_log, y2, 1.0)), y2);
    const real lin = fmadd(a * i21, e2 - e1, e1);
    const real fb = sel(ends_log, vexp(sel(ends_log, lin, 0.0)), lin);
    y = sel(outside, fb, y);
  }
  return y;
}

// ---- emission: measurement times against the step log, likelihood sums ---------------------------
struct Emitter {
  int io;            // measurement times emitted so far
  int base;          // trajectory-global index of log entry 0 (entries dropped by earlier flushes)
  bool floored;
  int status;
  real ll0, ll1, ll2, nneg;
};

TRPL_FN void emitter_init(Emitter& e) {
  e.io = 0; e.base = 0; e.floored = false; e.status = ST_OK;
  e.ll0 = splat(0.0); e.ll1 = splat(0.0); e.ll2 = splat(0.0); e.nneg = splat(0.0);
}

TRPL_FN void emitter_accumulate(Emitter& e, const TrajIn& in, bool want_ll, const ivec& k, const mask& take, const real& y) {
  if (in.curve) scatter(in.curve, k, take, y);
  if (want_ll && !in.post_pass) {
    e.nneg = e.nneg + sel(mand(take, y < 0.0), 1.0, 0.0);
    const real vk = gather(in.vals, k, take, 0.0);
    const real uk = gather(in.uncs, k, take, 1.0);
    const real r = (vlog10(vabs(y)) + in.scale_shift) - vk;
    const real r2 = r * r;
    const real u2 = 2.0 * (uk * uk);
    e.ll0 = e.ll0 + sel(take, r2 * rcp(in.s2T[0] + u2), 0.0);
    e.ll1 = e.ll1 + sel(take, r2 * rcp(in.s2T[1] + u2), 0.0);
    e.ll2 = e.ll2 + sel(take, r2 * rcp(in.s2T[2] + u2), 0.0);
  }
}

TRPL_FN void emitter_finish(Emitter& e, const TrajIn& in, bool want_ll, TrajMid& mid) {
  const int n_t = in.md->n_t;
  const ivec lane = lane_id();
  while (e.io < n_t) {                              // floor reached or integrator failure
    const ivec k = iadd(lane, e.io);
    emitter_accumulate(e, in, want_ll, k, k < n_t, splat(in.md->min_y));
    e.io += LANES;
  }
  if (want_ll && !in.post_pass) {
    mid.l[0] = -uni(warp_sum(e.ll0)); mid.l[1] = -uni(warp_sum(e.ll1)); mid.l[2] = -uni(warp_sum(e.ll2));
    mid.n_neg = uni(warp_sum(e.nneg));
  } else {
    mid.l[0] = mid.l[1] = mid.l[2] = 0.0; mid.n_neg = 0.0;
  }
}

// Deferred emission.  The integration loop only appends (t, S, dS/dt) of every accepted step to a
// per-warp log; this routine evaluates the measurement times the log covers, 32 at a time: every
// lane finds the step that contains its time by bisection of the log, interpolates
// (hermite_lane), applies the min_y floor (forward_solver.py:190-192: from the first value below
// min_y on, the curve IS min_y) and accumulates the likelihood sums.  It is deliberately NOT
// inlined: the interpolation and likelihood arithmetic (log, exp, log10, gathers, ballots) then
// cannot disturb the register allocation of the hot loop, and nothing it needs is live there.
// With `carry` (the log is full, the trajectory goes on) the last two entries move to the front
// so that later times can still see the two step points before their own step.
TRPL_NOINLINE void emit_history(const TrajIn& in, bool want_ll, double* hist, int n, Emitter& e, bool carry) {
  const MeasDesc& md = *in.md;
  const int n_t = md.n_t;
  const ivec lane = lane_id();
  const double t_last = (n > 0) ? hist[3 * (n - 1)] : -1.0;
  while (n > 0 && e.io < n_t && !e.floored) {
    const ivec k = iadd(lane, e.io);
    const mask in_range = k < n_t;
    const real tq = gather(in.times, k, in_range, DBL_MAX);
    const lanebits bits = warp_ballot(mand(in_range, tq <= t_last));
    if (bits == 0u) break;
    int cnt = 0;
    { lanebits b = bits; while (b & 1u) { ++cnt; b >>= 1; } }     // times ascend: the ready lanes are a prefix
    const mask take = lane < cnt;
    const real tqe = sel(take, tq, t_last);                        // idle lanes: a harmless exact hit
    // newest point of the containing step: the first log entry with t >= tq
    ivec pos = isplat(-1);
    for (int step = HIST_CAP / 2; step > 0; step >>= 1) {
      const ivec cand = iadd(pos, step);
      const mask ok = cand < n;
      const real tc = gather(hist, imul(cand, 3), ok, DBL_MAX);
      pos = seli(mand(ok, tc < tqe), cand, pos);
    }
    const ivec i2 = iclamp(iadd(pos, 1), 0, n - 1);
    const ivec i1 = iclamp(iadd(i2, -1), 0, n - 1), i0 = iclamp(iadd(i2, -2), 0, n - 1);
    const mask all = mconst(true);
    const real t2 = gather(hist, imul(i2, 3), all, 0.0), y2 = gather(hist, iadd(imul(i2, 3), 1), all, 0.0),
               s2 = gather(hist, iadd(imul(i2, 3), 2), all, 0.0);
    const real t1 = gather(hist, imul(i1, 3), all, 0.0), y1 = gather(hist, iadd(imul(i1, 3), 1), all, 0.0),
               s1 = gather(hist, iadd(imul(i1, 3), 2), all, 0.0);
    const real t0 = gather(hist, imul(i0, 3), all, 0.0), y0 = gather(hist, iadd(imul(i0, 3), 1), all, 0.0),
               s0 = gather(hist, iadd(imul(i0, 3), 2), all, 0.0);
    const ivec g = iadd(i2, e.base);                               // global index of the step's end point
    // lanes with fewer than two points (g == 0: the initial state) or an exact hit take the logged value
    const mask two = mand(g >= 1, i2 >= 1);
    real y = hermite_lane(tqe, mand(g >= 2, i2 >= 2), t0, y0, s0, sel(two, t1, t2 - 1.0), y1, s1, t2, y2, s2);
    y = sel(mor(mnot(two), tqe >= t2), y2, y);
    const lanebits low = warp_ballot(mand(take, y < md.min_y));
    if (low != 0u) {
      int firstlow = 0; { lanebits b = low; while (!(b & 1u)) { ++firstlow; b >>= 1; } }
      y = sel(lane >= firstlow, md.min_y, y);
      e.floored = true; e.status |= ST_FLOORED;
    }
    emitter_accumulate(e, in, want_ll, k, take, y);
    e.io += cnt;
    if (cnt < LANES) break;
  }
  if (carry && n >= 4) {
    const real v = gather(hist, iadd(lane, 3 * (n - 2)), lane < 6, 0.0);
    warp_sync();
    scatter(hist, lane, lane < 6, v);
    warp_sync();
    e.base += n - 2;
  }
}

// append one accepted step to the log (flushing it when full); returns true once the floor was hit
TRPL_FN bool log_point(const TrajIn& in, bool want_ll, Emitter& em, int& nh, double t, double val, double dval) {
  if (nh == HIST_CAP) {
    warp_sync();
    emit_history(in, want_ll, in.hist, nh, em, true);
    nh = 2;
    if (em.floored) return true;
  }
  const ivec lane = lane_id();
  scatter(in.hist, iadd(lane, 3 * nh), lane < 3, sel(lane == 0, t, sel(lane == 1, val, dval)));
  ++nh;
  return false;
}

// ---- stage combinations with compile-time coefficients ---------------------------------------
// After stage S-1 (0-based) has produced K_{S-1} (`kk`, still in registers; older increments come
// back from shared memory) build the argument and the c-combination of stage S:
//     us = u + sum_{p<S} a_Sp K_p ,   cs = sum_{p<S} (c_Sp / h) K_p .
// One instantiation per stage: the coefficients are immediates, every load is issued up front and
// there is no loop control (the generic loop cost 10% of the kernel in branches and constant loads).
template <int S, int P, int NPL, int MODEL>
TRPL_FN void combine_term(const Vec<NPL, MODEL>& kp, double ih, Vec<NPL, MODEL>& us, Vec<NPL, MODEL>& cs) {
  constexpr double a = Rodas4::A[S][P];
  const double cc = Rodas4::C[S][P] * ih;
  TRPL_UNROLL for (int j = 0; j < NPL; ++j) {
    if constexpr (S != 5) {       // stage 6's argument is built from stage 5's (stage_combine)
      us.n[j] = fmadd(a, kp.n[j], us.n[j]); us.q[j] = fmadd(a, kp.q[j], us.q[j]);
      if (MODEL == MODEL_TRAPS) us.t[j] = fmadd(a, kp.t[j], us.t[j]);
    }
    cs.n[j] = fmadd(cc, kp.n[j], cs.n[j]); cs.q[j] = fmadd(cc, kp.q[j], cs.q[j]);
    if (MODEL == MODEL_TRAPS) cs.t[j] = fmadd(cc, kp.t[j], cs.t[j]);
  }
}
template <int S, int NPL, int MODEL>
TRPL_FN void stage_combine(TrajMem& mem, double ih, const Vec<NPL, MODEL>& u, const Vec<NPL, MODEL>& kk,
                           Vec<NPL, MODEL>& us, Vec<NPL, MODEL>& cs) {
  typedef Slots<NPL, MODEL> SL;
  // Older increments come back from their memory through two buffers: the load of term p+1 is in
  // flight while term p is consumed.
  KRun<NPL, MODEL> ka, kb;
  Vec<NPL, MODEL> kp;
  if constexpr (S >= 2) {
    fence_stage_stores<NPL, MODEL>(mem);
    load_stage_nowait<0, NPL, MODEL>(mem, ka);
  }
  {
    // the newest increment is still in registers
    constexpr double a = Rodas4::A[S][S - 1];
    const double cc = Rodas4::C[S][S - 1] * ih;
    TRPL_UNROLL for (int j = 0; j < NPL; ++j) {
      if constexpr (S == 5) {
        // row 6 of A is row 5 plus e_5: the argument of stage 6 is the argument of stage 5 (still
        // in `us`) plus K_5
        us.n[j] = us.n[j] + kk.n[j]; us.q[j] = us.q[j] + kk.q[j];
        if (MODEL == MODEL_TRAPS) us.t[j] = us.t[j] + kk.t[j];
      } else {
        us.n[j] = fmadd(a, kk.n[j], u.n[j]); us.q[j] = fmadd(a, kk.q[j], u.q[j]);
        if (MODEL == MODEL_TRAPS) us.t[j] = fmadd(a, kk.t[j], u.t[j]);
      }
      cs.n[j] = cc * kk.n[j]; cs.q[j] = cc * kk.q[j];
      if (MODEL == MODEL_TRAPS) cs.t[j] = cc * kk.t[j];
    }
  }
  if constexpr (S >= 2) {
    wait_stage<0, NPL, MODEL>(mem);
    if constexpr (S >= 3) load_stage_nowait<1, NPL, MODEL>(mem, kb);
    unpack_k<NPL, MODEL>(ka, kp);
    combine_term<S, 0, NPL, MODEL>(kp, ih, us, cs);
  }
  if constexpr (S >= 3) {
    wait_stage<1, NPL, MODEL>(mem);
    if constexpr (S >= 4) load_stage_nowait<2, NPL, MODEL>(mem, ka);
    unpack_k<NPL, MODEL>(kb, kp);
    combine_term<S, 1, NPL, MODEL>(kp, ih, us, cs);
  }
  if constexpr (S >= 4) {
    wait_stage<2, NPL, MODEL>(mem);
    if constexpr (S >= 5) load_stage_nowait<3, NPL, MODEL>(mem, kb);
    unpack_k<NPL, MODEL>(ka, kp);
    combine_term<S, 2, NPL, MODEL>(kp, ih, us, cs);
  }
  if constexpr (S >= 5) {
    wait_stage<3, NPL, MODEL>(mem);
    unpack_k<NPL, MODEL>(kb, kp);
    combine_term<S, 3, NPL, MODEL>(kp, ih, us, cs);
  }
  // Row 6 of A is row 5 plus e_5, so the new state is (argument of stage 6) + K_6.  K_1..K_5 are
  // dead once this combination is formed: park the stage-6 argument in K_1's slot instead of
  // rebuilding it from five increments at the end of the step.
  if constexpr (S == 5) store_stage<NPL, MODEL>(mem, 0, us);
}
// ---- the trajectory -------------------------------------------------------------------------
// Control flow is a small state machine so that the right-hand side, the readout/emit block and the
// linear solve each exist at exactly ONE code site (the kernel is instruction-cache sensitive):
//   PH_ACCEPTED  evaluate f(u) at the newly accepted state, read the signal out, emit measurement
//                times, then start a step (Jacobian + factorisation), stage 1 uses f(u)
//   PH_STAGE     evaluate f(stage argument), add the c-combination, solve
//   PH_RETRY     step rejected: same u, new h; f(u) is re-evaluated (rejections are ~0.5% of the
//                steps, and this keeps f(u) out of registers and shared memory)
enum Phase { PH_ACCEPTED = 0, PH_STAGE = 1, PH_RETRY = 2 };

// K = W^{-1} r with the factorisation of this step (traps: occupancy condensed out, see the
// factorisation in run_trajectory)
template <int NPL, int MODEL, class PF>
TRPL_FN void stage_solve(TrajMem& mem, PF& pf, const Vec<NPL, MODEL>& r, Vec<NPL, MODEL>& kk) {
  typedef Slots<NPL, MODEL> SL;
  LaneMem& sm = mem.sm;
  if (MODEL != MODEL_TRAPS) kk.t[0] = splat(0.0);
  V2 b[NPL];
  if (MODEL == MODEL_TRAPS) {
    real w[NPL], gn[NPL], fnt[NPL], fqt[NPL], fqtn[NPL];
    real tr[6 * NPL];
    mem_wait_st(trmem<SL>(mem));
    mem_ld_pairs<3 * NPL>(trmem<SL>(mem), SL::TRAP, tr);
    mem_wait_ld(trmem<SL>(mem));
    TRPL_UNROLL for (int j = 0; j < NPL; ++j) {
      gn[j] = tr[6 * j + 1]; fnt[j] = tr[6 * j + 2]; fqt[j] = tr[6 * j + 3]; fqtn[j] = tr[6 * j + 4];
      w[j] = tr[6 * j + 0] * r.t[j];                        // idt * r_T
    }
    const real w_next = shfl_down(w[0], 1);
    TRPL_UNROLL for (int j = 0; j < NPL; ++j) {
      const real wn = (j == NPL - 1) ? w_next : w[j + 1];
      b[j].x = fmadd(fnt[j], w[j], r.n[j]);
      b[j].y = fmadd(fqt[j], w[j], fmadd(fqtn[j], wn, r.q[j]));
    }
    bt_solve<NPL>(b, fmem<SL>(mem), SL::FAC, sm, SL::XCH, pf);
    TRPL_UNROLL for (int j = 0; j < NPL; ++j) kk.t[j] = fmadd(gn[j], b[j].x, w[j]);
  } else {
    TRPL_UNROLL for (int j = 0; j < NPL; ++j) { b[j].x = r.n[j]; b[j].y = r.q[j]; }
    bt_solve<NPL>(b, fmem<SL>(mem), SL::FAC, sm, SL::XCH, pf);
  }
  TRPL_UNROLL for (int j = 0; j < NPL; ++j) { kk.n[j] = b[j].x; kk.q[j] = b[j].y; }
}

template <int NPL, int MODEL>
TRPL_FN bool is_nonstiff(const Coef& c, const NodeMask<NPL>& m, const Vec<NPL, MODEL>& u, double tend);   // explicit.h

// Returns true (and does nothing else) when `allow_defer` is set and the trajectory is classified
// non-stiff at t = 0: the caller hands it to the explicit Runge-Kutta path instead.
template <int NPL, int MODEL, bool FULL>
TRPL_FN bool run_trajectory(const TrajIn& in, const SolverOpts& opt, TrajMem& mem, TrajOut& out,
                            TrajMid& mid, bool allow_defer) {
  LaneMem& sm = mem.sm;
  typedef Slots<NPL, MODEL> SL;
  typedef Vec<NPL, MODEL> V;
  const MeasDesc& md = *in.md;
  const int L = md.nx;
  // The coefficients are formed once, parked in the uniform shared-memory slot and re-fetched by
  // each block of the loop that needs them (broadcast loads), instead of pinning registers.
  const Coef c = make_coef(in.par, md.thickness, L);
  park_coef(sm, SL::UNI, c);
  const NodeMask<NPL> m = make_mask<NPL, FULL>(L);
  const ivec lane = lane_id();
  const ivec node0 = imul(lane, NPL);
  const int n_t = md.n_t;
  const bool want_ll = !(opt.flags & OPT_NO_LIKELIHOOD);
  // min_y floor and IRF convolution need the whole curve: likelihood in a final pass over it
  const double min_y = md.min_y;

  // ---- initial condition (forward_solver.py:100-122) ----
  V u;
  double ex_floor = 0.0;            // error-control floor of the excess density (EXCESS_RANGE x initial peak)
  {
    real rho_run = splat(0.0);
    real dn_max = splat(0.0);
    real qloc[NPL];
    TRPL_UNROLL for (int j = 0; j < NPL; ++j) {
      const ivec i = iadd(node0, j);
      real dn;
      if (md.ini_mode == 0) {
        dn = gather(in.profile, i, m.real_node[j], 0.0) * 1e-21;
      } else {
        const double fluence = md.ini_a * in.fl_mult * 1e-14;
        const double alpha = md.ini_b * in.al_mult * 1e-7;
        const double x0 = 0.5 * c.dx;
        const double step = (L > 1) ? (md.thickness - c.dx) / (L - 1) : 0.0;   // np.linspace, sim_utils.py:269
        const real idx = to_real((md.ini_dir < 0) ? irsub(L - 1, i) : i);
        const real x = fmadd(idx, step, x0);
        dn = (fluence * alpha) * vexp(-(alpha * x));
      }
      dn_max = vmax(dn_max, sel(m.real_node[j], vabs(dn), 0.0));
      const real n = dn + c.n0, p = dn + c.p0;
      const real rho = (p - c.p0) - (n - c.n0);                  // forward_solver.py:28-29
      rho_run = rho_run + sel(m.real_node[j], rho, 0.0);
      qloc[j] = rho_run;
      u.n[j] = sel(m.real_node[j], n, 1.0);
      if (MODEL == MODEL_TRAPS) u.t[j] = splat(0.0);
    }
    if (MODEL != MODEL_TRAPS) u.t[0] = splat(0.0);
    // Gauss's law: running net charge = in-lane running sum + exclusive warp scan of lane totals
    ex_floor = EXCESS_RANGE * uni(warp_max(dn_max));
    const real incl = warp_scan_incl(rho_run);
    const real excl = incl - rho_run;
    TRPL_UNROLL for (int j = 0; j < NPL; ++j) u.q[j] = sel(m.real_node[j], qloc[j] + excl, 0.0);
  }

  const double tend = in.times[n_t - 1];
  if (allow_defer && is_nonstiff<NPL, MODEL>(c, m, u, tend)) return true;

  // ---- bookkeeping ----
  double t = 0.0;
  int status = ST_OK, n_acc = 0, n_rej = 0;
  int nh = 0;                       // entries in the history buffer
  Emitter em;                       // lives in local memory: only the (cold) emission touches it
  emitter_init(em);

  double h = 0.0, h_new = 0.0, gi = 0.0, ih = 0.0;
  float err2_old = 1e-8f;           // squared error norm of the last accepted step (floored at 1e-4)
  double ih_acc = 0.0;              // 1 / (size of the last accepted step)
  bool first = true, last_rejected = false, final_step = false;
  const double inv_n = 1.0 / (2.0 * L + ((MODEL == MODEL_TRAPS) ? L : 0));
  const double h_min = 1e-14 * fmax(tend, 1e-300);
  int phase = PH_ACCEPTED;
  int s = 0;
  V us = u;       // argument of the next right-hand-side evaluation
  V cs;           // sum_j c_sj / h K_j of the current stage
  TRPL_UNROLL for (int j = 0; j < NPL; ++j) { cs.n[j] = splat(0.0); cs.q[j] = splat(0.0); }
  TRPL_UNROLL for (int j = 0; j < (MODEL == MODEL_TRAPS ? NPL : 1); ++j) cs.t[j] = splat(0.0);
  typename PmChoice<SL>::type pf = PmChoice<SL>::make(mem);

  for (;;) {
    V r;
    RhsAux<NPL> aux;                // of the latest right-hand side; the Jacobian reuses it at stage 1
    {
      // PH_RETRY re-evaluates f(u) (us == u): rejections are rare (~0.5% of steps) and this keeps
      // f(u) out of shared memory
      const Coef cr = fetch_coef(sm, SL::UNI);
      rhs<NPL, MODEL>(cr, m, us, r, aux);
      if (phase == PH_ACCEPTED) {
        // ---- newly accepted state (us == u): read the signal out and log it ----
        double val, dval;
        readout<NPL, MODEL>(cr, m, md.meas_type, u, r, aux, val, dval);
        if (log_point(in, want_ll, em, nh, t, val, dval)) break;
        // done when the last measurement time is reached, or the signal fell through its floor
        // (forward_solver.py:190-192: the rest of the curve is min_y by definition)
        if (t >= tend || val < min_y) break;
        if (n_acc == 0) {
          // ---- initial step (Hairer's d0/d1 rule on the scaled norms) ----
          real s0 = splat(0.0), s1 = splat(0.0);
          TRPL_UNROLL for (int j = 0; j < NPL; ++j) {
            const real iscn = rcp(fmadd(opt.rtol, vabs(u.n[j]), opt.atol));
            const real iscq = rcp(fmadd(opt.rtol, vmax(vabs(u.n[j]), vabs(aux.p[j])), opt.atol));
            const real a = u.n[j] * iscn, b = r.n[j] * iscn, q = u.q[j] * iscq, g = r.q[j] * iscq;
            s0 = s0 + sel(m.real_node[j], fmadd(a, a, q * q), 0.0);
            s1 = s1 + sel(m.real_node[j], fmadd(b, b, g * g), 0.0);
          }
          const double d0 = sqrt(uni(warp_sum(s0))), d1 = sqrt(uni(warp_sum(s1)));
          h = (d1 > 0.0 && d0 > 0.0) ? 0.01 * d0 / d1 : 1e-6;
          h = fmin(h, 1e-3 * fmax(tend, 1e-300));
          if (!(h > 0.0)) h = 1e-6;
        } else {
          h = h_new;
        }
      }
    }
    if (phase != PH_STAGE) {
      // ---- start (or restart) a step from u with step size h; stage 1 right-hand side is f(u) ----
      if (n_acc + n_rej >= opt.max_steps) { status |= ST_MAX_STEPS; break; }
      if (opt.hmax > 0.0) h = fmin(h, opt.hmax);
      final_step = false;
      if (t + 1.01 * h >= tend) { h = tend - t; final_step = true; }
      if (h < h_min) { status |= ST_H_UNDERFLOW; break; }
      ih = uni(rcp(splat(h)));
      gi = (1.0 / RODAS4_GAMMA) * ih;
      {
        // W = 1/(gamma h) I - J, factorised
        Blk A[NPL], B[NPL], C[NPL];
        JacTraps<NPL> jt;
        jacobian<NPL, MODEL>(fetch_coef(sm, SL::UNI), m, u, aux, A, B, C, jt);
        TRPL_UNROLL for (int j = 0; j < NPL; ++j) {
          A[j] = blk_neg(A[j]); C[j] = blk_neg(C[j]);
          B[j].a00 = gi - B[j].a00; B[j].a01 = -B[j].a01; B[j].a10 = -B[j].a10; B[j].a11 = gi - B[j].a11;
        }
        // the front contact has no left neighbour (Q_0 is the fixed corner field)
        A[0] = blk_sel(m.first_lane, blk_zero(), A[0]);
        if (MODEL == MODEL_TRAPS) {
          // condense the node-local trap occupancy out of the block rows
          real g_n[NPL];
          real tr[6 * NPL];
          TRPL_UNROLL for (int j = 0; j < NPL; ++j) {
            const real idt = rcp(gi - jt.ft_t[j]);
            g_n[j] = jt.ft_n[j] * idt;              // K_T = idt * r_T + g_n * K_N
            tr[6 * j + 0] = idt; tr[6 * j + 1] = g_n[j];
            tr[6 * j + 2] = jt.fn_t[j]; tr[6 * j + 3] = jt.fq_t[j];
            tr[6 * j + 4] = jt.fq_tn[j]; tr[6 * j + 5] = jt.fq_tn[j];
          }
          mem_st_pairs<3 * NPL>(trmem<SL>(mem), SL::TRAP, tr);
          const real gn_next = shfl_down(g_n[0], 1);
          TRPL_UNROLL for (int j = 0; j < NPL; ++j) {
            const real gnn = (j == NPL - 1) ? gn_next : g_n[j + 1];
            B[j].a00 = B[j].a00 - jt.fn_t[j] * g_n[j];
            B[j].a10 = B[j].a10 - jt.fq_t[j] * g_n[j];
            C[j].a10 = C[j].a10 - jt.fq_tn[j] * gnn;
          }
        }
        bt_factor<NPL>(A, B, C, fmem<SL>(mem), SL::FAC, sm, SL::XCH_FACTOR, pf);
      }
      s = 0;
    } else {
      TRPL_UNROLL for (int j = 0; j < NPL; ++j) {
        r.n[j] = r.n[j] + cs.n[j]; r.q[j] = r.q[j] + cs.q[j];
        if (MODEL == MODEL_TRAPS) r.t[j] = r.t[j] + cs.t[j];
      }
    }

    // ---- K_s = W^{-1} r ----
    V kk;
    stage_solve<NPL, MODEL>(mem, pf, r, kk);

    if (s < 5) {
      // ---- keep K_s, build the next stage argument and c-combination ----
      if (s < 4) store_stage<NPL, MODEL>(mem, s, kk);     // K_5 is consumed from registers only
      ++s;
      switch (s) {
        case 1: stage_combine<1, NPL, MODEL>(mem, ih, u, kk, us, cs); break;
        case 2: stage_combine<2, NPL, MODEL>(mem, ih, u, kk, us, cs); break;
        case 3: stage_combine<3, NPL, MODEL>(mem, ih, u, kk, us, cs); break;
        case 4: stage_combine<4, NPL, MODEL>(mem, ih, u, kk, us, cs); break;
        default: stage_combine<5, NPL, MODEL>(mem, ih, u, kk, us, cs); break;
      }
      phase = PH_STAGE;
      continue;
    }

    // ---- stage 6 done: u_new = u + sum_j m_j K_j = (stage-6 argument, parked by stage_combine<5>)
    // + K_6; the error estimate is K_6 ----
    {
      KRun<NPL, MODEL> parked;
      fence_stage_stores<NPL, MODEL>(mem);
      load_stage_nowait<0, NPL, MODEL>(mem, parked);
      wait_stage<0, NPL, MODEL>(mem);
      unpack_k<NPL, MODEL>(parked, us);
    }
    TRPL_UNROLL for (int j = 0; j < NPL; ++j) {
      us.n[j] = us.n[j] + kk.n[j]; us.q[j] = us.q[j] + kk.q[j];
      if (MODEL == MODEL_TRAPS) us.t[j] = us.t[j] + kk.t[j];
    }
    // error norm: the scales only steer the step size, so their reciprocals are the 2^-23 hardware
    // seed and the max() has no NaN bookkeeping (non-finite states are caught by `bad`)
    real esum = splat(0.0);
    mask bad = mconst(false);
    real pold[NPL];
    const Coef ce = fetch_coef(sm, SL::UNI);
    holes<NPL, MODEL>(ce, m, u, pold);
    TRPL_UNROLL for (int j = 0; j < NPL; ++j) {
      // The density error is measured relative to the EXCESS density N - n0 (floored at ex_floor):
      // the signal is n0 dP + p0 dN + dN dP, so once the excess has fallen below the dark density a
      // scale rtol |N| would stop controlling the only thing the readout sees (DESIGN.md section 2).
      // The charge keeps the larger carrier density at the old state as its scale (the cheaper bound
      // N + |p0 - n0| let one of 24576 benchmark trajectories slip to 1.6e-5).
      const real mx = vmax_fast(vmax_fast(vabs(u.n[j] - ce.n0), vabs(us.n[j] - ce.n0)), ex_floor);
      const real mq = vmax_fast(vabs(u.n[j]), vabs(pold[j]));
      const real iscn = rcp_approx(fmadd(opt.rtol, mx, opt.atol));
      const real iscq = rcp_approx(fmadd(opt.rtol, mq, opt.atol));
      const real en = kk.n[j] * iscn, eq = kk.q[j] * (iscq * Q_ERR_WEIGHT);
      real e2 = fmadd(en, en, eq * eq);
      if (MODEL == MODEL_TRAPS) {
        const real isct = rcp_approx(fmadd(opt.rtol, vmax_fast(vabs(u.t[j]), vmax_fast(vabs(us.t[j]), mx)), opt.atol));
        const real et = kk.t[j] * isct;
        e2 = fmadd(et, et, e2);
      }
      esum = esum + sel(m.real_node[j], e2, 0.0);
      bad = mor(bad, mand(m.real_node[j], mor(is_nan(us.n[j]), is_nan(us.q[j]))));
    }
    const double err2 = uni(warp_sum(esum)) * inv_n;            // err^2
    const bool nonfinite = warp_any(bad) || !(err2 == err2) || err2 > 1e300;

    // ---- controller (Hairer's RODAS: standard + Gustafsson predictive) ----
    // Single precision, no divisions or square roots: with e2 = err^2 the standard factor is
    //   h_new / h = 0.9 err^(-1/4) = 0.9 e2^(-1/8)           clamped to [1/6, 5],
    // the predictive one (after an accepted step of size h_acc with error err_old)
    //   h_new / h = 0.9 (h / h_acc) (err_old / err^2)^(1/4) = 0.9 (h / h_acc) e2^(-1/4) e2_old^(1/8),
    // and the smaller of the two is taken.
    const float e2f = nonfinite ? 1e20f : (float)fmax(fmin(err2, 1e30), 1e-30);
    float ifac = fmaxf(1.0f / 6.0f, fminf(5.0f, CTL_SAFETY * ctl_powf(e2f, -0.125f)));
    h_new = h * (double)ifac;
    if (!nonfinite && err2 <= 1.0) {
      ++n_acc;
      if (!first) {
        float ifg = CTL_SAFETY * (float)(h * ih_acc) * ctl_powf(e2f, -0.25f) * ctl_powf(err2_old, 0.125f);
        ifg = fmaxf(1.0f / 6.0f, fminf(5.0f, ifg));
        ifac = fminf(ifac, ifg);
        h_new = h * (double)ifac;
      }
      first = false; ih_acc = ih; err2_old = fmaxf(1e-4f, e2f);
      if (last_rejected) h_new = fmin(h_new, h);
      last_rejected = false;
      t = final_step ? tend : t + h;
      TRPL_UNROLL for (int j = 0; j < NPL; ++j) {
        u.n[j] = us.n[j]; u.q[j] = us.q[j];
        if (MODEL == MODEL_TRAPS) u.t[j] = us.t[j];
      }
      phase = PH_ACCEPTED;
    } else {
      ++n_rej;
      last_rejected = true;
      h = nonfinite ? 0.1 * h : h_new;
      TRPL_UNROLL for (int j = 0; j < NPL; ++j) {
        us.n[j] = u.n[j]; us.q[j] = u.q[j];
        if (MODEL == MODEL_TRAPS) us.t[j] = u.t[j];
      }
      phase = PH_RETRY;
    }
  }
  // replay the logged steps: measurement times, floor, likelihood sums; anything not reached
  // (floor, or integrator failure) is min_y: forward_solver.py:168 + :190-192
  warp_sync();
  emit_history(in, want_ll, in.hist, nh, em, false);
  emitter_finish(em, in, want_ll, mid);
  out.status = status | em.status; out.n_acc = n_acc; out.n_rej = n_rej;
  return false;
}

// ---- likelihood (trial_move_evaluation.py:117-166): streaming sums, or a pass over the curve ----
TRPL_FN void finalize_trajectory(const TrajIn& in, const TailIn& tl, const SolverOpts& opt,
                                 const TrajMid& mid, TrajOut& out) {
  const bool want_ll = !(opt.flags & OPT_NO_LIKELIHOOD);
  const int n_t = in.md->n_t;
  if (want_ll) {
    double l[3];
    double n_neg;
    int n_c = n_t;
    bool ok = true;
    const bool ladder = in.post_pass && (opt.flags & OPT_LADDER) && tl.ladder_n > 0 && tl.r2_scratch;
    if (in.post_pass) {
      warp_sync();
      const double* sol = in.curve;
      if (tl.irf.nk > 0) {
        ok = irf_convolve_trim(in.times, in.curve, n_t, tl.irf, n_c);
        sol = tl.irf.trim;
        if (!ok) out.status |= ST_CONV_FAIL;
      }
      if (ok) array_loglik(sol, n_c, in.vals, in.uncs, in.scale_shift, in.s2T,
                           (opt.flags & OPT_FORCE_MIN_Y) != 0, l, n_neg,
                           ladder ? tl.r2_scratch : nullptr, ladder ? tl.u2_scratch : nullptr, nullptr);
    } else {
      l[0] = mid.l[0]; l[1] = mid.l[1]; l[2] = mid.l[2];
      n_neg = mid.n_neg;
    }
    const double ninf = -HUGE_VAL;
    if (!ok) {
      l[0] = l[1] = l[2] = ninf;
    } else {
      if (!(n_neg < 0.2 * n_c)) { out.status |= ST_NEG_FRAC; l[0] = l[1] = l[2] = ninf; }
      if (l[0] != l[0]) { out.status |= ST_NAN_LL; l[0] = ninf; }
      if (l[1] != l[1]) l[1] = ninf;
      if (l[2] != l[2]) l[2] = ninf;
    }
    out.logll[0] = l[0]; out.logll[1] = l[1]; out.logll[2] = l[2];
    if (ladder) {
      const bool failed = !ok || !(n_neg < 0.2 * n_c);
      ladder_loglik(tl.r2_scratch, tl.u2_scratch, failed ? 0 : n_c, in.s2T[1], tl.ladder_T, tl.ladder_n,
                    tl.ladder_out, failed);
    }
  } else {
    out.logll[0] = out.logll[1] = out.logll[2] = 0.0;
  }
}

// ---- fitted curve (OPT_FIT): what the likelihood compared, point by point ----------------------
// From the trajectory's stored signal (in.curve, complete once its trajectory kernel is done), by
// the routines finalize_trajectory uses: the IRF convolution and trim, then array_loglik, which
// writes log10(|y|, floored) + scale_shift for the n_c compared points.  The streaming sums of
// emitter_accumulate form the same value from the same y (the curve holds it bit for bit, with the
// min_y floor applied), so fit[k] - vals[k] is the residual of every path.  Points past n_c are
// NaN; all of them when the convolution failed.  Run as its own pass so that nothing of it is
// compiled into the trajectory kernels.
TRPL_FN void fit_trajectory(const TrajIn& in, const TailIn& tl, const SolverOpts& opt, double* fit) {
  const int n_t = in.md->n_t;
  int n_c = n_t;
  bool ok = true;
  const double* sol = in.curve;
  if (tl.irf.nk > 0) {
    ok = irf_convolve_trim(in.times, in.curve, n_t, tl.irf, n_c);
    sol = tl.irf.trim;
  }
  if (!ok) n_c = 0;
  if (n_c > 0) {
    double l[3], n_neg;
    array_loglik(sol, n_c, in.vals, in.uncs, in.scale_shift, in.s2T, (opt.flags & OPT_FORCE_MIN_Y) != 0, l, n_neg,
                 nullptr, nullptr, fit);
  }
  const ivec lane = lane_id();
  for (int k0 = n_c; k0 < n_t; k0 += LANES) {
    const ivec k = iadd(lane, k0);
    scatter(fit, k, k < n_t, splat(NAN));
  }
  warp_sync();
}

}  // namespace trpl
