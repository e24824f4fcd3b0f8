// extrapolation.h - the low-latency integrator: extrapolated linearly implicit Euler (Deuflhard's
// SEULEX scheme: Hairer & Wanner, Solving ODEs II, sec. IV.9), six columns of the harmonic sequence,
// order 6, with the columns of one step spread over the four warps of a CTA.
//
// Why a second integrator.  A parallel-tempering iteration is as slow as its slowest trajectory, and
// with RODAS4 (trajectory.h) a trajectory is 400-900 steps of six stages that can only run one after
// the other: 6.5 us per step whether one warp or a whole CTA works on it (DESIGN.md section 5).  An
// extrapolation step from u over H computes, for j = 1..6, j linearly implicit Euler steps of size
// H/j,
//     (j/H I - J(u)) d_m = f(y_m),  y_{m+1} = y_m + d_m,   T_j = y_j,
// and combines the six results with fixed weights (Aitken-Neville for an expansion in H/j).  The
// columns are INDEPENDENT of each other.  Given to the warps as {6}, {5}, {4, 1}, {3, 2}, no warp
// runs more than six solves per step - the depth of one RODAS4 step - while the step is of order 6
// instead of 4 and 3.5-4.2x longer at the same accuracy (measured on the fixture states at rtol 1e-7:
// 69 / 123 / 147 / 107 steps against 240 / 520 / 593 / 434, curves at the measurement times within
// 7e-6 of the converged ones through the same dense output).  Total work is 21 solves + 6
// factorisations per step, about 1.25x RODAS4's per unit of time, so this is the integrator for
// SMALL batches (tempering); the throughput path stays RODAS4.
//
// Everything below the step is shared with trajectory.h: right-hand side, exact Jacobian,
// block-tridiagonal factorisation and solve, error scales, step log, dense output, likelihood.
// Two drivers:
//   run_trajectory_seulex      one warp runs all six columns in turn (host lock-step build: the CPU
//                              test tier; also a device kernel, for bit-for-bit comparison)
//   run_trajectory_seulex_cta  four warps, columns in parallel, results exchanged through shared
//                              memory once per step (device only)
// Both accumulate the six increments in the same fixed order with the same operations, so they
// produce identical bits.
#pragma once
#include "explicit.h"

namespace trpl {
using namespace simt;

struct Seulex {
  static constexpr int K = 6;
  // order in which the columns are combined: 6 | 5 | 4 1 | 3 2, and which warp computes which: warp w
  // runs order(group_first(w)) .. order(group_first(w + 1) - 1).  A column costs one factorisation
  // (about 3.5 solves) plus j solves and right-hand sides, so {6}, {5}, {4, 1}, {3, 2} is the
  // grouping with the shortest longest chain (13.5 solve-equivalents; {6}, {5,1}, {4,2}, {3}: 14.8).
  TRPL_FN static constexpr int order(int ci) { return ci == 0 ? 6 : ci == 1 ? 5 : ci == 2 ? 4 : ci == 3 ? 1 : ci == 4 ? 3 : 2; }
  TRPL_FN static constexpr int group_first(int w) { return w == 0 ? 0 : w == 1 ? 1 : w == 2 ? 2 : w == 3 ? 4 : 6; }
  // T_66 = sum_j A_j T_j and T_66 - T_65 = sum_j B_j T_j for the harmonic sequence (Lagrange weights
  // of the polynomial in H/j at 0; exact rationals, tools/proto/seulex_weights.py); sum A = 1, sum B = 0
  TRPL_FN static constexpr double A(int j) {
    return j == 1 ? -1.0 / 120.0 : j == 2 ? 4.0 / 3.0 : j == 3 ? -81.0 / 4.0 : j == 4 ? 256.0 / 3.0
         : j == 5 ? -3125.0 / 24.0 : 324.0 / 5.0;
  }
  TRPL_FN static constexpr double B(int j) {
    return j == 1 ? -1.0 / 120.0 : j == 2 ? 2.0 / 3.0 : j == 3 ? -27.0 / 4.0 : j == 4 ? 64.0 / 3.0
         : j == 5 ? -625.0 / 24.0 : 54.0 / 5.0;
  }
  // T_55 - T_54 = sum_j B5_j T_j: the error estimate one order down.  In the asymptotic regime it is
  // 14-25x the order-6 estimate at an accepted step; where the Jacobian changes character inside a
  // step (SRH lifetime collapsing from tauP to tauN as the injection falls through p0: state 13 of
  // the staub fixture) the order-6 difference can be accidentally small while this one jumps.  The
  // step is judged by max(err_6, err_5 / ERR5_RATIO).
  TRPL_FN static constexpr double B5(int j) {
    return j == 1 ? 1.0 / 24.0 : j == 2 ? -4.0 / 3.0 : j == 3 ? 27.0 / 4.0 : j == 4 ? -32.0 / 3.0
         : j == 5 ? 125.0 / 24.0 : 0.0;
  }
};
#ifndef TRPL_SEULEX_ERR5_RATIO
#define TRPL_SEULEX_ERR5_RATIO 20.0
#endif
// Nonlinearity monitor.  All columns of a step use the Jacobian of its START, and both difference
// estimates are blind to a change of regime the start does not announce (same SRH knee: a step of
// 73 ns at tau_S = 90 ns was accepted with err 0.5 and is 1e-3 off).  A step is therefore also
// rejected (and halved) when the signal's logarithmic decay rate -dS/dt / S at its end differs from
// the one at its start by more than this factor; on single-exponential decays it never triggers.
#ifndef TRPL_SEULEX_RATE_CHANGE
#define TRPL_SEULEX_RATE_CHANGE 1.25
#endif

// true when the step u -> us changed the signal's decay rate by more than TRPL_SEULEX_RATE_CHANGE
template <int NPL, int MODEL>
TRPL_FN bool seulex_regime_changed(const Coef& c, const NodeMask<NPL>& m, int meas_type, const Vec<NPL, MODEL>& us,
                                   double val0, double dval0, double val_floor) {
  Vec<NPL, MODEL> f1;
  RhsAux<NPL> aux1;
  rhs<NPL, MODEL>(c, m, us, f1, aux1);
  double val1, dval1;
  readout<NPL, MODEL>(c, m, meas_type, us, f1, aux1, val1, dval1);
  if (!(val0 > 0.0) || !(val1 > val_floor) || !(dval0 < 0.0) || !(dval1 < 0.0)) return false;
  const double r = (dval1 * val0) / (dval0 * val1);          // rate at the end / rate at the start
  return r > TRPL_SEULEX_RATE_CHANGE || r * TRPL_SEULEX_RATE_CHANGE < 1.0;
}
#ifndef TRPL_SEULEX_SAFETY
#define TRPL_SEULEX_SAFETY 0.9f
#endif
// The local tolerance is this fraction of rtol: with steps of about one e-fold of the signal a local
// error of rtol per step leaves 2-5e-5 on the fast-decaying fixture curves (RODAS4 at the same rtol:
// 4e-6); at 0.3 rtol both are within 1e-5 of the converged curves, for 20% more steps.
#ifndef TRPL_SEULEX_TOL_FACTOR
#define TRPL_SEULEX_TOL_FACTOR 0.3
#endif
// Steps are also capped at this many e-folds of the signal: the dense output (quintic Hermite of
// ln S through the step's ends and the point before, trajectory.h) is only as good as the step is
// short against the time scale of the signal, and an order-6 step can span several e-folds.
#ifndef TRPL_SEULEX_EFOLDS
#define TRPL_SEULEX_EFOLDS 1.0
#endif

template <int NPL, int MODEL>
TRPL_FN void vec_zero(Vec<NPL, MODEL>& v) {
  TRPL_UNROLL for (int j = 0; j < NPL; ++j) { v.n[j] = splat(0.0); v.q[j] = splat(0.0); }
  TRPL_UNROLL for (int j = 0; j < (MODEL == MODEL_TRAPS ? NPL : 1); ++j) v.t[j] = splat(0.0);
}
// y = a + b
template <int NPL, int MODEL>
TRPL_FN void vec_add(const Vec<NPL, MODEL>& a, const Vec<NPL, MODEL>& b, Vec<NPL, MODEL>& y) {
  TRPL_UNROLL for (int j = 0; j < NPL; ++j) {
    y.n[j] = a.n[j] + b.n[j]; y.q[j] = a.q[j] + b.q[j];
    if (MODEL == MODEL_TRAPS) y.t[j] = a.t[j] + b.t[j];
  }
  if (MODEL != MODEL_TRAPS) y.t[0] = splat(0.0);
}
// y += w x
template <int NPL, int MODEL>
TRPL_FN void vec_axpy(double w, const Vec<NPL, MODEL>& x, Vec<NPL, MODEL>& y) {
  TRPL_UNROLL for (int j = 0; j < NPL; ++j) {
    y.n[j] = fmadd(w, x.n[j], y.n[j]); y.q[j] = fmadd(w, x.q[j], y.q[j]);
    if (MODEL == MODEL_TRAPS) y.t[j] = fmadd(w, x.t[j], y.t[j]);
  }
}

// W = gi I - J(u), factorised into the trajectory's storage (the block run_trajectory has inline)
template <int NPL, int MODEL, class PF>
TRPL_FN void factor_shifted(double gi, const Coef& c, const NodeMask<NPL>& m, const Vec<NPL, MODEL>& u,
                            const RhsAux<NPL>& aux, TrajMem& mem, PF& pf) {
  typedef Slots<NPL, MODEL> SL;
  Blk A[NPL], B[NPL], C[NPL];
  JacTraps<NPL> jt;
  jacobian<NPL, MODEL>(c, m, u, aux, A, B, C, jt);
  TRPL_UNROLL for (int j = 0; j < NPL; ++j) {
    A[j] = blk_neg(A[j]); C[j] = blk_neg(C[j]);
    B[j].a00 = gi - B[j].a00; B[j].a01 = -B[j].a01; B[j].a10 = -B[j].a10; B[j].a11 = gi - B[j].a11;
  }
  A[0] = blk_sel(m.first_lane, blk_zero(), A[0]);       // the front contact has no left neighbour
  if (MODEL == MODEL_TRAPS) {
    real g_n[NPL];
    real tr[6 * NPL];
    TRPL_UNROLL for (int j = 0; j < NPL; ++j) {
      const real idt = rcp(gi - jt.ft_t[j]);
      g_n[j] = jt.ft_n[j] * idt;
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
  bt_factor<NPL>(A, B, C, fmem<SL>(mem), SL::FAC, mem.sm, SL::XCH_FACTOR, pf);
}

// Column j: j linearly implicit Euler steps of size H/j from u with the Jacobian at u; returns the
// increment D_j = T_j - u.  f(u) is re-evaluated here (it also yields what the Jacobian reuses), so
// nothing of the step's start has to stay live across the columns.
template <int NPL, int MODEL, class PF>
TRPL_FN void seulex_column(int j, double ih, const NodeMask<NPL>& m, const Vec<NPL, MODEL>& u, TrajMem& mem,
                           PF& pf, Vec<NPL, MODEL>& d) {
  typedef Slots<NPL, MODEL> SL;
  typedef Vec<NPL, MODEL> V;
  const double gi = (double)j * ih;
  V r;
  {
    RhsAux<NPL> aux;
    const Coef c = fetch_coef(mem.sm, SL::UNI);
    rhs<NPL, MODEL>(c, m, u, r, aux);
    factor_shifted<NPL, MODEL>(gi, c, m, u, aux, mem, pf);
  }
  vec_zero<NPL, MODEL>(d);
  for (int mm = 0; mm < j; ++mm) {
    if (mm > 0) {
      V y;
      vec_add<NPL, MODEL>(u, d, y);
      RhsAux<NPL> aux;
      rhs<NPL, MODEL>(fetch_coef(mem.sm, SL::UNI), m, y, r, aux);
    }
    V kk;
    stage_solve<NPL, MODEL>(mem, pf, r, kk);
    TRPL_UNROLL for (int i = 0; i < NPL; ++i) {
      d.n[i] = d.n[i] + kk.n[i]; d.q[i] = d.q[i] + kk.q[i];
      if (MODEL == MODEL_TRAPS) d.t[i] = d.t[i] + kk.t[i];
    }
  }
}

// squared error norm of the estimate `de` for the step u -> us: the scales of trajectory.h
template <int NPL, int MODEL>
TRPL_FN double seulex_err2(const SolverOpts& opt, const Coef& c, const NodeMask<NPL>& m, const Vec<NPL, MODEL>& u,
                           const Vec<NPL, MODEL>& us, const Vec<NPL, MODEL>& de, double ex_floor, double inv_n,
                           bool& nonfinite) {
  real esum = splat(0.0);
  mask bad = mconst(false);
  real pold[NPL];
  holes<NPL, MODEL>(c, m, u, pold);
  const double rtol = TRPL_SEULEX_TOL_FACTOR * opt.rtol;
  TRPL_UNROLL for (int j = 0; j < NPL; ++j) {
    const real mx = vmax_fast(vmax_fast(vabs(u.n[j] - c.n0), vabs(us.n[j] - c.n0)), ex_floor);
    const real mq = vmax_fast(vabs(u.n[j]), vabs(pold[j]));
    const real iscn = rcp_approx(fmadd(rtol, mx, opt.atol));
    const real iscq = rcp_approx(fmadd(rtol, mq, opt.atol));
    const real en = de.n[j] * iscn, eq = de.q[j] * (iscq * Q_ERR_WEIGHT);
    real e2 = fmadd(en, en, eq * eq);
    if (MODEL == MODEL_TRAPS) {
      const real isct = rcp_approx(fmadd(rtol, vmax_fast(vabs(u.t[j]), vmax_fast(vabs(us.t[j]), mx)), opt.atol));
      const real et = de.t[j] * isct;
      e2 = fmadd(et, et, e2);
    }
    esum = esum + sel(m.real_node[j], e2, 0.0);
    bad = mor(bad, mand(m.real_node[j], mor(is_nan(us.n[j]), is_nan(us.q[j]))));
  }
  const double err2 = uni(warp_sum(esum)) * inv_n;
  nonfinite = warp_any(bad) || !(err2 == err2) || err2 > 1e300;
  return err2;
}

// step-size factor of an order-6 step from its squared error norm (err^(-1/6) = e2^(-1/12))
TRPL_FN float seulex_factor(double err2, bool nonfinite) {
  const float e2f = nonfinite ? 1e20f : (float)fmax(fmin(err2, 1e30), 1e-30);
  return fmaxf(0.1f, fminf(4.0f, TRPL_SEULEX_SAFETY * ctl_powf(e2f, -1.0f / 12.0f)));
}

// initial step size: the d0/d1 rule of trajectory.h
template <int NPL, int MODEL>
TRPL_FN double seulex_first_step(const SolverOpts& opt, const NodeMask<NPL>& m, const Vec<NPL, MODEL>& u,
                                 const Vec<NPL, MODEL>& f, const RhsAux<NPL>& aux, double tend) {
  real s0 = splat(0.0), s1 = splat(0.0);
  TRPL_UNROLL for (int j = 0; j < NPL; ++j) {
    const real iscn = rcp(fmadd(opt.rtol, vabs(u.n[j]), opt.atol));
    const real iscq = rcp(fmadd(opt.rtol, vmax(vabs(u.n[j]), vabs(aux.p[j])), opt.atol));
    const real a = u.n[j] * iscn, b = f.n[j] * iscn, q = u.q[j] * iscq, g = f.q[j] * iscq;
    s0 = s0 + sel(m.real_node[j], fmadd(a, a, q * q), 0.0);
    s1 = s1 + sel(m.real_node[j], fmadd(b, b, g * g), 0.0);
  }
  const double d0 = sqrt(uni(warp_sum(s0))), d1 = sqrt(uni(warp_sum(s1)));
  double h = (d1 > 0.0 && d0 > 0.0) ? 0.01 * d0 / d1 : 1e-6;
  h = fmin(h, 1e-3 * fmax(tend, 1e-300));
  if (!(h > 0.0)) h = 1e-6;
  return h;
}

// ---- driver 1: one warp, all columns in turn -------------------------------------------------
template <int NPL, int MODEL, bool FULL>
TRPL_FN void run_trajectory_seulex(const TrajIn& in, const SolverOpts& opt, TrajMem& mem, TrajOut& out,
                                   TrajMid& mid) {
  typedef Slots<NPL, MODEL> SL;
  typedef Vec<NPL, MODEL> V;
  LaneMem& sm = mem.sm;
  const MeasDesc& md = *in.md;
  const int L = md.nx;
  const NodeMask<NPL> m = make_mask<NPL, FULL>(L);
  const bool want_ll = !(opt.flags & OPT_NO_LIKELIHOOD);
  const double min_y = md.min_y;
  V u;
  double ex_floor;
  {
    const Coef c = make_coef(in.par, md.thickness, L);
    park_coef(sm, SL::UNI, c);
    initial_state<NPL, MODEL>(in, c, m, u);
    real dn_max = splat(0.0);
    TRPL_UNROLL for (int j = 0; j < NPL; ++j) dn_max = vmax(dn_max, sel(m.real_node[j], vabs(u.n[j] - c.n0), 0.0));
    ex_floor = EXCESS_RANGE * uni(warp_max(dn_max));
  }
  const double tend = in.times[md.n_t - 1];
  const double inv_n = 1.0 / (2.0 * L + ((MODEL == MODEL_TRAPS) ? L : 0));
  const double h_min = 1e-14 * fmax(tend, 1e-300);
  double t = 0.0, h = 0.0, h_new = 0.0, h_cap = 0.0, val0 = 0.0, dval0 = 0.0, val_floor = 0.0;
  int status = ST_OK, n_acc = 0, n_rej = 0, nh = 0;
  bool last_rejected = false, done = false;
  Emitter em;
  emitter_init(em);
  typename PmChoice<SL>::type pf = PmChoice<SL>::make(mem);

  while (!done) {
    {
      // newly accepted (or initial) state: signal, its time derivative, step log
      V f0;
      RhsAux<NPL> aux;
      const Coef c = fetch_coef(sm, SL::UNI);
      rhs<NPL, MODEL>(c, m, u, f0, aux);
      double val, dval;
      readout<NPL, MODEL>(c, m, md.meas_type, u, f0, aux, val, dval);
      val0 = val; dval0 = dval;
      if (n_acc == 0) val_floor = fmax(min_y, EXCESS_RANGE * val);     // below: rounding noise, no monitor
      if (log_point(in, want_ll, em, nh, t, val, dval)) break;
      if (t >= tend || val < min_y) break;
      h = (n_acc == 0) ? seulex_first_step<NPL, MODEL>(opt, m, u, f0, aux, tend) : h_new;
      // (no cap once the signal is below the controlled dynamic range: nothing is claimed there)
      h_cap = (dval != 0.0 && val > val_floor) ? TRPL_SEULEX_EFOLDS * fabs(val / dval) : tend;
    }
    for (;;) {
      if (n_acc + n_rej >= opt.max_steps) { status |= ST_MAX_STEPS; done = true; break; }
      h = fmin(h, h_cap);
      if (opt.hmax > 0.0) h = fmin(h, opt.hmax);
      bool final_step = false;
      if (t + 1.01 * h >= tend) { h = tend - t; final_step = true; }
      if (h < h_min) { status |= ST_H_UNDERFLOW; done = true; break; }
      const double ih = uni(rcp(splat(h)));
      V du, de, de5;
      vec_zero<NPL, MODEL>(du);
      vec_zero<NPL, MODEL>(de);
      vec_zero<NPL, MODEL>(de5);
      for (int ci = 0; ci < Seulex::K; ++ci) {
        const int j = Seulex::order(ci);
        V d;
        seulex_column<NPL, MODEL>(j, ih, m, u, mem, pf, d);
        vec_axpy<NPL, MODEL>(Seulex::A(j), d, du);
        vec_axpy<NPL, MODEL>(Seulex::B(j), d, de);
        vec_axpy<NPL, MODEL>(Seulex::B5(j), d, de5);
      }
      V us;
      vec_add<NPL, MODEL>(u, du, us);
      bool nonfinite, nonfinite5;
      double err2 = seulex_err2<NPL, MODEL>(opt, fetch_coef(sm, SL::UNI), m, u, us, de, ex_floor, inv_n, nonfinite);
      const double err2_5 = seulex_err2<NPL, MODEL>(opt, fetch_coef(sm, SL::UNI), m, u, us, de5, ex_floor, inv_n, nonfinite5);
      err2 = fmax(err2, err2_5 * (1.0 / (TRPL_SEULEX_ERR5_RATIO * TRPL_SEULEX_ERR5_RATIO)));
      nonfinite = nonfinite || nonfinite5;
      const float ifac = seulex_factor(err2, nonfinite);
      h_new = h * (double)ifac;
      if (!nonfinite && err2 <= 1.0 && h > 16.0 * h_min &&
          seulex_regime_changed<NPL, MODEL>(fetch_coef(sm, SL::UNI), m, md.meas_type, us, val0, dval0, val_floor)) {
        ++n_rej;
        last_rejected = true;
        h = 0.5 * h;
        continue;
      }
      if (!nonfinite && err2 <= 1.0) {
        ++n_acc;
        if (last_rejected) h_new = fmin(h_new, h);
        last_rejected = false;
        t = final_step ? tend : t + h;
        u = us;
        break;
      }
      ++n_rej;
      last_rejected = true;
      h = nonfinite ? 0.1 * h : h_new;
    }
  }
  warp_sync();
  emit_history(in, want_ll, in.hist, nh, em, false);
  emitter_finish(em, in, want_ll, mid);
  out.status = status | em.status; out.n_acc = n_acc; out.n_rej = n_rej;
}

// Exchange area of the cooperative driver, behind the four warps' slices of shared memory: the
// column increments as double2 (N, Q) [column][node][lane] and, for traps, their T components as
// double [column][node][lane] behind those.  'std' keeps two such buffers, alternating by step
// parity, and needs ONE __syncthreads per step.  Traps keeps one and adds a second __syncthreads once
// every warp has read it: at 4 nodes per lane that is 18 432 B instead of 36 864, the CTA with its four
// 23 040 B slices is 110.6 KB, and two CTAs still share an SM (2 x 129 KB would not fit its 228 KB).
template <int NPL, int MODEL>
struct SeulexXch {
  static constexpr int PER_BUF = Seulex::K * NPL * 32;       // entries of each component array
  static constexpr int BUFS = (MODEL == MODEL_TRAPS) ? 1 : 2;
  static constexpr int BYTES = BUFS * PER_BUF * ((MODEL == MODEL_TRAPS) ? 16 + 8 : 16);
};

#if defined(__CUDACC__) && !defined(TRPL_HOST_EMU)
// ---- driver 2: four warps of a CTA, columns in parallel ----------------------------------------
// xch: SeulexXch<NPL, MODEL>; s_flag: one int of shared memory for the rare step-log flush.  Every
// warp holds the full state (lane l owns the same nodes in all four), computes its own columns, and
// after a __syncthreads combines all six increments in the fixed order of the one-warp driver -
// identical bits, identical decisions.
template <int NPL, int MODEL, bool FULL>
__device__ __forceinline__ void run_trajectory_seulex_cta(const TrajIn& in, const SolverOpts& opt, TrajMem& mem,
                                                          double2* xch, int* s_flag, int warp, TrajOut& out,
                                                          TrajMid& mid) {
  typedef Slots<NPL, MODEL> SL;
  typedef Vec<NPL, MODEL> V;
  typedef SeulexXch<NPL, MODEL> XC;
  LaneMem& sm = mem.sm;
  const MeasDesc& md = *in.md;
  const int L = md.nx;
  const int lane = threadIdx.x & 31;
  const NodeMask<NPL> m = make_mask<NPL, FULL>(L);
  const bool want_ll = !(opt.flags & OPT_NO_LIKELIHOOD);
  const double min_y = md.min_y;
  V u;
  double ex_floor;
  {
    const Coef c = make_coef(in.par, md.thickness, L);
    park_coef(sm, SL::UNI, c);
    initial_state<NPL, MODEL>(in, c, m, u);
    real dn_max = splat(0.0);
    TRPL_UNROLL for (int j = 0; j < NPL; ++j) dn_max = vmax(dn_max, sel(m.real_node[j], vabs(u.n[j] - c.n0), 0.0));
    ex_floor = EXCESS_RANGE * uni(warp_max(dn_max));
  }
  const double tend = in.times[md.n_t - 1];
  const double inv_n = 1.0 / ((MODEL == MODEL_TRAPS) ? 3.0 * L : 2.0 * L);   // the one-warp driver's value
  const double h_min = 1e-14 * fmax(tend, 1e-300);
  double t = 0.0, h = 0.0, h_new = 0.0, h_cap = 0.0, val0 = 0.0, dval0 = 0.0, val_floor = 0.0;
  int status = ST_OK, n_acc = 0, n_rej = 0, nh = 0, buf = 0;
  bool last_rejected = false, done = false;
  Emitter em;
  emitter_init(em);
  typename PmChoice<SL>::type pf = PmChoice<SL>::make(mem);
  constexpr int PER_BUF = XC::PER_BUF;
  double* const xt = reinterpret_cast<double*>(xch + PER_BUF);      // traps: the T components

  while (!done) {
    {
      V f0;
      RhsAux<NPL> aux;
      const Coef c = fetch_coef(sm, SL::UNI);
      rhs<NPL, MODEL>(c, m, u, f0, aux);
      double val, dval;
      readout<NPL, MODEL>(c, m, md.meas_type, u, f0, aux, val, dval);
      val0 = val; dval0 = dval;
      if (n_acc == 0) val_floor = fmax(min_y, EXCESS_RANGE * val);     // below: rounding noise, no monitor
      // the step log belongs to warp 0; every warp counts its entries
      if (nh == HIST_CAP) {
        if (warp == 0) {
          warp_sync();
          emit_history(in, want_ll, in.hist, nh, em, true);
          if (lane == 0) *s_flag = em.floored ? 1 : 0;
        }
        __syncthreads();
        nh = 2;
        const int floored = *s_flag;
        __syncthreads();
        if (floored) break;
      }
      if (warp == 0 && lane < 3) in.hist[3 * nh + lane] = (lane == 0) ? t : (lane == 1 ? val : dval);
      ++nh;
      if (t >= tend || val < min_y) break;
      h = (n_acc == 0) ? seulex_first_step<NPL, MODEL>(opt, m, u, f0, aux, tend) : h_new;
      // (no cap once the signal is below the controlled dynamic range: nothing is claimed there)
      h_cap = (dval != 0.0 && val > val_floor) ? TRPL_SEULEX_EFOLDS * fabs(val / dval) : tend;
    }
    for (;;) {
      if (n_acc + n_rej >= opt.max_steps) { status |= ST_MAX_STEPS; done = true; break; }
      h = fmin(h, h_cap);
      if (opt.hmax > 0.0) h = fmin(h, opt.hmax);
      bool final_step = false;
      if (t + 1.01 * h >= tend) { h = tend - t; final_step = true; }
      if (h < h_min) { status |= ST_H_UNDERFLOW; done = true; break; }
      const double ih = uni(rcp(splat(h)));
      double2* xb = xch + buf * PER_BUF;
      for (int ci = Seulex::group_first(warp); ci < Seulex::group_first(warp + 1); ++ci) {
        V d;
        seulex_column<NPL, MODEL>(Seulex::order(ci), ih, m, u, mem, pf, d);
        TRPL_UNROLL for (int i = 0; i < NPL; ++i) {
          xb[(ci * NPL + i) * 32 + lane] = make_double2(d.n[i], d.q[i]);
          if (MODEL == MODEL_TRAPS) xt[(ci * NPL + i) * 32 + lane] = d.t[i];
        }
      }
      __syncthreads();
      V du, de, de5;
      vec_zero<NPL, MODEL>(du);
      vec_zero<NPL, MODEL>(de);
      vec_zero<NPL, MODEL>(de5);
      TRPL_UNROLL for (int ci = 0; ci < Seulex::K; ++ci) {
        const int j = Seulex::order(ci);
        V d;
        TRPL_UNROLL for (int i = 0; i < NPL; ++i) {
          const double2 v = xb[(ci * NPL + i) * 32 + lane];
          d.n[i] = v.x; d.q[i] = v.y;
          if (MODEL == MODEL_TRAPS) d.t[i] = xt[(ci * NPL + i) * 32 + lane];
        }
        if (MODEL != MODEL_TRAPS) d.t[0] = 0.0;
        vec_axpy<NPL, MODEL>(Seulex::A(j), d, du);
        vec_axpy<NPL, MODEL>(Seulex::B(j), d, de);
        vec_axpy<NPL, MODEL>(Seulex::B5(j), d, de5);
      }
      if (XC::BUFS == 1) __syncthreads();      // one buffer: read by every warp before the next columns write it
      else buf ^= 1;
      V us;
      vec_add<NPL, MODEL>(u, du, us);
      bool nonfinite, nonfinite5;
      double err2 = seulex_err2<NPL, MODEL>(opt, fetch_coef(sm, SL::UNI), m, u, us, de, ex_floor, inv_n, nonfinite);
      const double err2_5 = seulex_err2<NPL, MODEL>(opt, fetch_coef(sm, SL::UNI), m, u, us, de5, ex_floor, inv_n, nonfinite5);
      err2 = fmax(err2, err2_5 * (1.0 / (TRPL_SEULEX_ERR5_RATIO * TRPL_SEULEX_ERR5_RATIO)));
      nonfinite = nonfinite || nonfinite5;
      const float ifac = seulex_factor(err2, nonfinite);
      h_new = h * (double)ifac;
      if (!nonfinite && err2 <= 1.0 && h > 16.0 * h_min &&
          seulex_regime_changed<NPL, MODEL>(fetch_coef(sm, SL::UNI), m, md.meas_type, us, val0, dval0, val_floor)) {
        ++n_rej;
        last_rejected = true;
        h = 0.5 * h;
        continue;
      }
      if (!nonfinite && err2 <= 1.0) {
        ++n_acc;
        if (last_rejected) h_new = fmin(h_new, h);
        last_rejected = false;
        t = final_step ? tend : t + h;
        u = us;
        break;
      }
      ++n_rej;
      last_rejected = true;
      h = nonfinite ? 0.1 * h : h_new;
    }
  }
  __syncthreads();
  if (warp == 0) {
    emit_history(in, want_ll, in.hist, nh, em, false);
    emitter_finish(em, in, want_ll, mid);
    out.status = status | em.status; out.n_acc = n_acc; out.n_rej = n_rej;
  }
}
#endif

}  // namespace trpl
