// irf.h - instrument-response convolution and the final likelihood pass over a stored curve.
//
// Replaces, per trajectory and inside the kernel,
//   laplace.py:44-86    do_irf_convolution (resample to dt_irf/2, moment convolution, max-shift)
//   laplace.py:178-222  convolve
//   laplace.py:89-129   post_conv_trim (cut to the convolved span, interpolate back)
//   utils.py:16-32      set_min_y
//   trial_move_evaluation.py:117-166  negative test, log10 residuals, weighted sum
// The moment tables (laplace.py:13-41, make_I_tables) are a one-off host precompute
// (metrotrpl_b200/laplace.py) uploaded with the problem.
//
// Work is spread over the lanes (resampled points, convolution outputs and measurement times are
// independent); the three scratch arrays live in a per-warp slice of global memory that stays in L2.
#pragma once
#include <float.h>
#include "simt.h"

namespace trpl {
using namespace simt;

struct IrfDesc {
  const double* mom;   // [nk][3] moment integrals I_m^n
  int nk;              // rows of the table (= IRF samples); 0 = no convolution for this measurement
  double dt;           // mean IRF time step
  double* ry;          // scratch: resampled curve           [n_rs]
  double* hk;          // scratch: convolved curve           [nk_conv + 1]
  double* trim;        // scratch: convolved curve on the measurement times [n_t]
};

// points of a curve ending at tend resampled to dt/2: len(np.arange(0, tend + dt/4, dt/2))
TRPL_HD int irf_resample_count(double tend, double dt) { return (int)ceil((tend + dt / 4) / (dt / 2)); }

// np.interp(x, xp, fp) for one x per lane, xp ascending, xp[0] <= x <= xp[n-1]
TRPL_FN real interp_lanes(const double* xp, const double* fp, int n, const real& x, const mask& take) {
  ivec lo = isplat(0);
  // Measurement times are usually equally spaced: guess the interval from the mean spacing and keep
  // the guess if it brackets x (xp[g] <= x < xp[g+1], or g is the last interval); that IS the
  // interval the search below would return.  Any miss nearby: everyone searches.
  bool searched = n < 3;
  if (!searched) {
    const double inv = (double)(n - 1) / (xp[n - 1] - xp[0]);
    const ivec g = iclamp(to_int_floor((x - xp[0]) * inv), 0, n - 2);
    const real xg = gather(xp, g, take, 0.0), xg1 = gather(xp, iadd(g, 1), take, 1.0);
    const mask hit = mand(xg <= x, mor(x < xg1, g == n - 2));
    if (local_any(mand(take, mnot(hit)))) searched = true; else lo = g;
  }
  if (searched) {
    ivec hi = isplat(n - 1);
    lo = isplat(0);
    // invariant xp[lo] <= x; find the largest such lo (uniform trip count)
    for (int span = n; span > 1; span = (span + 1) >> 1) {
      const ivec mid = ishr1(iaddv(iaddv(lo, hi), isplat(1)));
      const real xm = gather(xp, mid, take, 0.0);
      const mask le = xm <= x;
      lo = seli(le, mid, lo);
      hi = seli(le, hi, iadd(mid, -1));
    }
  }
  lo = iclamp(lo, 0, n - 2 > 0 ? n - 2 : 0);
  const ivec lo1 = iadd(lo, n > 1 ? 1 : 0);
  const real x0 = gather(xp, lo, take, 0.0), x1 = gather(xp, lo1, take, 1.0);
  const real y0 = gather(fp, lo, take, 0.0), y1 = gather(fp, lo1, take, 0.0);
  const real slope = (y1 - y0) / (x1 - x0);
  real y = slope * (x - x0) + y0;
  y = sel(x >= x1, y1, y);            // exact at the right end, as np.interp
  return y;
}

// Returns false when the reference would have failed the convolution (-> likelihood -inf).
// On success trim[0..n_c) holds the convolved, max-shifted signal on times[0..n_c).
TRPL_FN bool irf_convolve_trim(const double* times, const double* curve, int n_t, const IrfDesc& f,
                               int& n_c) {
  const ivec lane = lane_id();
  const double tend = times[n_t - 1];
  const double half = f.dt / 2;
  const int n_rs = irf_resample_count(tend, f.dt);
  if (n_rs < 3) return false;
  const int nk = (n_rs - 1) / 2;
  const int last_rs = n_rs - 1;
  // resampled abscissa j*half, the last one clamped to tend (laplace.py:68-72)
  const double x_last = fmin((double)last_rs * half, tend);

  // ---- 1. resample (laplace.py:68-74) ----
  mask any_nan = mconst(false);
  for (int j0 = 0; j0 < n_rs; j0 += LANES) {
    const ivec j = iadd(lane, j0);
    const mask take = j < n_rs;
    real x = to_real(j) * half;
    x = sel(j == last_rs, x_last, x);
    const real y = interp_lanes(times, curve, n_t, x, take);
    any_nan = mor(any_nan, mand(take, is_nan(y)));
    scatter(f.ry, j, take, y);
  }
  warp_sync();
  if (warp_any(any_nan)) return false;

  // ---- 2. moment convolution (laplace.py:178-222) ----
  // hk[k] = sum_{m < min(k, nk_irf)}  b(kp) I0_m + i1(kp) I1_m + i2(kp) I2_m ,   kp = k - 1 - m,
  //   b = ry[2kp+1],  i1 = ry[2kp+2] - ry[2kp],  i2 = 2 (ry[2kp+2] - 2 ry[2kp+1] + ry[2kp]).
  // Every lane owns OPL CONSECUTIVE outputs: the (b, i1, i2) triples of lag m+1 are those of lag m
  // shifted by one output, so each lag costs one new 128-bit load and one new triple per lane instead
  // of two loads and one triple per OUTPUT (the pass was a quarter of the nx = 256 kernel).  Each
  // output still sums its lags in ascending order with the same operations: same bits as before.
#ifndef TRPL_IRF_OPL
#define TRPL_IRF_OPL 4
#endif
  constexpr int OPL = TRPL_IRF_OPL;
  real best = splat(-DBL_MAX);
  ivec best_k = isplat(0x7fffffff);
  for (int kb = 0; kb <= nk; kb += OPL * LANES) {
    const ivec k0 = iadd(imul(lane, OPL), kb);                // first output of this lane
    const int k_max = kb + OPL * LANES - 1;
    const int m_hi = (k_max < f.nk) ? k_max : f.nk;           // lags needed by the largest k of this batch
    // window at lag 0: kp = k0 - 1 + j.  Triples of kp < 0 are zero (the lag does not exist for that
    // output); those of kp >= nk only feed outputs beyond nk, which are never stored.  Loads reach
    // kp = nk: ry[2 nk] closes the triple of nk - 1 (ry[2 nk + 1] may be the first word behind the
    // resampled curve, still inside the scratch slice, and is not used).
    real tb[OPL], t1[OPL], t2[OPL], acc[OPL];
    real a_new;                                               // ry[2 kp] of the newest (lowest) kp
    {
      real a[OPL + 1], b[OPL];
      TRPL_UNROLL for (int jj = 0; jj < OPL; ++jj) {
        const ivec kp = iadd(k0, jj - 1);
        gather2(f.ry, imul(kp, 2), mand(kp >= 0, kp <= nk), 0.0, a[jj], b[jj]);
      }
      { const ivec kp = iadd(k0, OPL - 1); a[OPL] = gather(f.ry, imul(kp, 2), mand(kp >= 1, kp <= nk), 0.0); }
      TRPL_UNROLL for (int jj = 0; jj < OPL; ++jj) {
        const ivec kp = iadd(k0, jj - 1);
        const mask ok = mand(kp >= 0, kp < nk);
        tb[jj] = sel(ok, b[jj], 0.0);
        t1[jj] = sel(ok, a[jj + 1] - a[jj], 0.0);
        t2[jj] = sel(ok, 2.0 * ((a[jj + 1] - 2.0 * b[jj]) + a[jj]), 0.0);
        acc[jj] = splat(0.0);
      }
      a_new = a[0];
    }
    TRPL_UNROLL4 for (int m = 0; m < m_hi; ++m) {
      const double m0 = f.mom[3 * m], m1 = f.mom[3 * m + 1], m2 = f.mom[3 * m + 2];
      // the triple that enters at the next lag: kp = k0 - 2 - m (its load is in flight during the sums)
      const ivec kpn = iadd(k0, -2 - m);
      const mask okn = mand(kpn >= 0, kpn < nk);
      real an, bn;
      gather2(f.ry, imul(kpn, 2), mand(kpn >= 0, kpn <= nk), 0.0, an, bn);
      TRPL_UNROLL for (int jj = 0; jj < OPL; ++jj)
        acc[jj] = acc[jj] + fmadd(t2[jj], m2, fmadd(t1[jj], m1, tb[jj] * m0));
      TRPL_UNROLL for (int jj = OPL - 1; jj > 0; --jj) { tb[jj] = tb[jj - 1]; t1[jj] = t1[jj - 1]; t2[jj] = t2[jj - 1]; }
      tb[0] = sel(okn, bn, 0.0);
      t1[0] = sel(okn, a_new - an, 0.0);
      t2[0] = sel(okn, 2.0 * ((a_new - 2.0 * bn) + an), 0.0);
      a_new = an;
    }
    TRPL_UNROLL for (int jj = 0; jj < OPL; ++jj) {
      const ivec k = iadd(k0, jj);
      const mask take = k <= nk;
      scatter(f.hk, k, take, acc[jj]);
      // running argmax, first occurrence (a lane's outputs ascend; ties across lanes: smallest k below)
      const mask better = mand(take, acc[jj] > best);
      best = sel(better, acc[jj], best);
      best_k = seli(better, k, best_k);
      any_nan = mor(any_nan, mand(take, is_nan(acc[jj])));
    }
  }
  warp_sync();
  if (warp_any(any_nan)) return false;
  // ---- 3. max-shift (laplace.py:80-84) ----
  const double vmax_all = uni(warp_max(best));
  const real cand = sel(best == vmax_all, to_real(best_k), 4e9);
  const int kmax = (int)uni(warp_min(cand));
  const double t_shift = (2 * kmax == last_rs) ? x_last : (double)(2 * kmax) * half;
  const double x_end = (2 * nk == last_rs) ? x_last : (double)(2 * nk) * half;
  const double max_ct = x_end - t_shift;                      // conv_t[-1]
  if (max_ct == 0.0) return false;

  // ---- 4. trim to the convolved span and interpolate back (laplace.py:119-127) ----
  real cnt = splat(0.0);
  for (int i0 = 0; i0 < n_t; i0 += LANES) {
    const ivec i = iadd(lane, i0);
    const mask take = i < n_t;
    const real te = gather(times, i, take, DBL_MAX);
    cnt = cnt + sel(mand(take, te < max_ct), 1.0, 0.0);
  }
  n_c = (int)uni(warp_sum(cnt));                              // times ascend: a prefix
  if (n_c < 1) return false;
  for (int i0 = 0; i0 < n_c; i0 += LANES) {
    const ivec i = iadd(lane, i0);
    const mask take = i < n_c;
    const real x = gather(times, i, take, 0.0);
    // conv_t[j] = fl(rt[2j] - t_shift); start from the arithmetic guess and fix the rounding
    ivec j = to_int_floor((x + t_shift) / f.dt);
    j = iclamp(j, 0, nk - 1);
    TRPL_UNROLL for (int fix = 0; fix < 2; ++fix) {
      const real tj = sel(imul(j, 2) == last_rs, x_last, to_real(imul(j, 2)) * half) - t_shift;
      j = seli(mand(tj > x, j > 0), iadd(j, -1), j);
    }
    TRPL_UNROLL for (int fix = 0; fix < 2; ++fix) {
      const ivec jn = iadd(j, 1);
      const real tn = sel(imul(jn, 2) == last_rs, x_last, to_real(imul(jn, 2)) * half) - t_shift;
      j = seli(mand(tn <= x, jn < nk), jn, j);
    }
    const ivec j1 = iadd(j, 1);
    const real x0 = sel(imul(j, 2) == last_rs, x_last, to_real(imul(j, 2)) * half) - t_shift;
    const real x1 = sel(imul(j1, 2) == last_rs, x_last, to_real(imul(j1, 2)) * half) - t_shift;
    const real y0 = gather(f.hk, j, take, 0.0), y1 = gather(f.hk, j1, take, 0.0);
    const real slope = (y1 - y0) / (x1 - x0);
    real y = slope * (x - x0) + y0;
    y = sel(x >= x1, y1, y);
    scatter(f.trim, i, take, y);
  }
  warp_sync();
  return true;
}

// Likelihood of a stored signal sol[0..n_c) against vals/uncs[0..n_c): abs/negative count,
// optional set_min_y floor, log10 residuals, three temperatures (trial_move_evaluation.py:117-166).
// fit_out (optional): the compared values log10(|sol|, floored) + shift, [n_c].
TRPL_FN void array_loglik(const double* sol, int n_c, const double* vals, const double* uncs,
                          double shift, const double* s2T, bool force_min_y, double* ll, double& n_neg,
                          double* r2_out, double* u2_out, double* fit_out) {
  const ivec lane = lane_id();
  int first_floor = n_c;
  double floor_y = 0.0;
  if (force_min_y) {
    // utils.py:16-32: raise |sol| to 10**min(vals - shift) from the index np.searchsorted finds on
    // -|sol| (a plain bisection, reproduced step for step)
    real mn = splat(DBL_MAX);
    for (int k0 = 0; k0 < n_c; k0 += LANES) {
      const ivec k = iadd(lane, k0);
      mn = vmin(mn, gather(vals, k, k < n_c, DBL_MAX) - shift);
    }
    floor_y = pow(10.0, uni(warp_min(mn)));
    int lo = 0, hi = n_c;
    while (lo < hi) {
      const int mid = lo + ((hi - lo) >> 1);
      if (-fabs(sol[mid]) < -floor_y) lo = mid + 1; else hi = mid;
    }
    first_floor = lo;
  }
  real l0 = splat(0.0), l1 = splat(0.0), l2 = splat(0.0), neg = splat(0.0);
  for (int k0 = 0; k0 < n_c; k0 += LANES) {
    const ivec k = iadd(lane, k0);
    const mask take = k < n_c;
    const real y = gather(sol, k, take, 1.0);
    neg = neg + sel(mand(take, y < 0.0), 1.0, 0.0);
    real ya = vabs(y);
    ya = sel(k >= first_floor, floor_y, ya);
    const real vk = gather(vals, k, take, 0.0);
    const real uk = gather(uncs, k, take, 1.0);
    const real f = vlog10(ya) + shift;
    if (fit_out) scatter(fit_out, k, take, f);
    const real r = f - vk;
    const real r2 = r * r;
    const real u2 = 2.0 * (uk * uk);
    l0 = l0 + sel(take, r2 * rcp(s2T[0] + u2), 0.0);
    l1 = l1 + sel(take, r2 * rcp(s2T[1] + u2), 0.0);
    l2 = l2 + sel(take, r2 * rcp(s2T[2] + u2), 0.0);
    if (r2_out) { scatter(r2_out, k, take, r2); scatter(u2_out, k, take, u2); }
  }
  ll[0] = -uni(warp_sum(l0)); ll[1] = -uni(warp_sum(l1)); ll[2] = -uni(warp_sum(l2));
  n_neg = uni(warp_sum(neg));
  if (r2_out) warp_sync();
}

// Likelihood of the same curve at every temperature of a tempering ladder:
//   ll(T_j) = - sum_k r2_k / (sigma^2 T_j + 2 u_k^2)      (trial_move_evaluation.py:150-156, ll_func(T))
// so that replica-exchange swaps (metropolis.py:66-90) never need a re-simulation.  Lanes take
// temperatures, the residuals are broadcast.
TRPL_FN void ladder_loglik(const double* r2, const double* u2, int n_c, double sigma2,
                           const double* temps, int n_T, double* out, bool failed) {
  const ivec lane = lane_id();
  for (int j0 = 0; j0 < n_T; j0 += LANES) {
    const ivec j = iadd(lane, j0);
    const mask take = j < n_T;
    const real s = sigma2 * gather(temps, j, take, 1.0);
    real acc = splat(0.0);
    for (int k = 0; k < n_c; ++k) acc = fmadd(splat(r2[k]), rcp(s + u2[k]), acc);
    real res = -acc;
    res = sel(is_nan(res), -HUGE_VAL, res);
    if (failed) res = splat(-HUGE_VAL);
    scatter(out, j, take, res);
  }
}

}  // namespace trpl
