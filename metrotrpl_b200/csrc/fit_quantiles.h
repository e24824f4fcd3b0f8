// fit_quantiles.h - the per-column arithmetic of trpl_fit_quantiles: exact, NaN-aware quantiles of
// each point of the fit buffer over the parameter sets of a run, equal bit for bit to
// np.nanquantile(fit, q, axis=0, method="linear") of NumPy 2.3.
//
// The order statistics are found by an MSB radix select on order-preserving 64-bit keys, 8 bits per
// pass: a target rank keeps the key prefix found so far and its rank among the values that share
// it; every pass histograms the next digit of those values, and qt_pick moves the target into the
// bucket that holds its rank.  After 8 passes the prefix is the key of the order statistic.
// fit_quantiles_kernel (trpl_kernels.cu) builds the histograms in shared memory; the host lock-step
// build (tests/emu/quantiles_emu.cpp) builds them in a loop and runs the same routines.
#pragma once
#include <math.h>
#include <stdint.h>
#include <string.h>
#include "../../include/metrotrpl_b200.h"
#include "simt.h"     // TRPL_FN

namespace {

constexpr int QT_DIGIT_BITS = 8;
constexpr int QT_BINS = 1 << QT_DIGIT_BITS;
constexpr int QT_PASSES = 64 / QT_DIGIT_BITS;
constexpr int QT_MAX_TARGETS = 2 * TRPL_MAX_QUANTILES;   // floor and floor + 1 of every level

// The arguments the caller passes; null or the message the call is refused with.
inline const char* qt_check(int n_q, const double* q) {
  if (n_q < 1 || n_q > TRPL_MAX_QUANTILES) return "trpl_fit_quantiles: n_q must be in 1..TRPL_MAX_QUANTILES (8)";
  if (!q) return "trpl_fit_quantiles: q is NULL";
  for (int j = 0; j < n_q; ++j)
    if (!(q[j] >= 0.0 && q[j] <= 1.0)) return "trpl_fit_quantiles: quantile levels must lie in [0, 1]";
  return nullptr;
}

TRPL_FN uint64_t qt_bits(double x) {
  uint64_t b;
  memcpy(&b, &x, sizeof b);
  return b;
}

TRPL_FN double qt_double(uint64_t b) {
  double x;
  memcpy(&x, &b, sizeof x);
  return x;
}

// Order-preserving key of a non-NaN double: -inf < ... < -0.0 < +0.0 < ... < +inf as unsigned keys.
TRPL_FN uint64_t qt_key(double x) {
  const uint64_t b = qt_bits(x), s = (uint64_t)1 << 63;
  return (b & s) ? ~b : (b | s);
}

TRPL_FN double qt_value(uint64_t k) {
  const uint64_t s = (uint64_t)1 << 63;
  return qt_double((k & s) ? (k ^ s) : ~k);
}

// Rounded IEEE operations, never contracted into an FMA (NumPy rounds every step).
#if defined(__CUDACC__) && !defined(TRPL_HOST_EMU)
TRPL_FN double qt_add(double a, double b) { return __dadd_rn(a, b); }
TRPL_FN double qt_sub(double a, double b) { return __dsub_rn(a, b); }
TRPL_FN double qt_mul(double a, double b) { return __dmul_rn(a, b); }
#else      // the host lock-step build compiles with -ffp-contract=off
TRPL_FN double qt_add(double a, double b) { return a + b; }
TRPL_FN double qt_sub(double a, double b) { return a - b; }
TRPL_FN double qt_mul(double a, double b) { return a * b; }
#endif

// NumPy's _quantile for method="linear" on n values: virtual index v = (n - 1) q; the neighbours
// floor(v) and floor(v) + 1, both clamped to n - 1 when v >= n - 1 (NumPy then takes index -1, and
// its gamma is v - (-1)); gamma = v - floor(v) otherwise.  n >= 1.
TRPL_FN void qt_ranks(int n, double q, int& lo, int& hi, double& gamma) {
  const double v = qt_mul((double)(n - 1), q);
  if (v >= (double)(n - 1)) {
    lo = hi = n - 1;
    gamma = qt_sub(v, -1.0);
  } else {
    const double f = floor(v);
    lo = (int)f;
    hi = lo + 1;
    gamma = qt_sub(v, f);
  }
}

// NumPy's _lerp: a + (b - a) t, or b - (b - a)(1 - t) where t >= 0.5.
TRPL_FN double qt_lerp(double a, double b, double t) {
  const double d = qt_sub(b, a);
  return t >= 0.5 ? qt_sub(b, qt_mul(d, qt_sub(1.0, t))) : qt_add(a, qt_mul(d, t));
}

// Inserts rank r into the ascending list rank[0..nt) unless it is there; returns the new length.
TRPL_FN int qt_insert(int* rank, int nt, int r) {
  int i = 0;
  while (i < nt && rank[i] < r) ++i;
  if (i < nt && rank[i] == r) return nt;
  for (int m = nt; m > i; --m) rank[m] = rank[m - 1];
  rank[i] = r;
  return nt + 1;
}

// The order statistics a column of n non-NaN values needs for levels q[0..n_q): ascending, no
// duplicates.  Returns how many (0 for n == 0).
TRPL_FN int qt_targets(int n, int n_q, const double* q, int* rank) {
  if (n < 1) return 0;
  int nt = 0;
  for (int j = 0; j < n_q; ++j) {
    int lo, hi;
    double g;
    qt_ranks(n, q[j], lo, hi, g);
    nt = qt_insert(rank, nt, lo);
    nt = qt_insert(rank, nt, hi);
  }
  return nt;
}

// One radix pass of one target: hist[QT_BINS] counts the digit of the values that share the target's
// prefix, rank is the target's rank among them.  Returns the digit of the bucket holding that rank
// and leaves rank as the rank inside the bucket.
TRPL_FN unsigned qt_pick(const uint32_t* hist, uint32_t& rank) {
  uint32_t below = 0;
  for (unsigned d = 0; d < (unsigned)QT_BINS; ++d) {
    const uint32_t c = hist[d];
    if (rank < below + c) { rank -= below; return d; }
    below += c;
  }
  return QT_BINS - 1;      // not reached: the ranks are below the values counted
}

// Shift of the digit of pass p, and whether key k shares prefix `pre` of the digits before it.
TRPL_FN int qt_shift(int p) { return 64 - QT_DIGIT_BITS * (p + 1); }
TRPL_FN bool qt_match(uint64_t k, uint64_t pre, int p) {
  return p == 0 || ((k ^ pre) >> (qt_shift(p) + QT_DIGIT_BITS)) == 0;
}

// Quantile q of a column of n non-NaN values (NaN for n == 0), from the keys key[0..nt) of its
// order statistics rank[0..nt) (qt_targets).
TRPL_FN double qt_finish(int n, double q, const int* rank, const uint64_t* key, int nt) {
  if (n < 1) return qt_double(0x7ff8000000000000ull);
  int lo, hi;
  double g;
  qt_ranks(n, q, lo, hi, g);
  double a = 0.0, b = 0.0;
  for (int i = 0; i < nt; ++i) {
    if (rank[i] == lo) a = qt_value(key[i]);
    if (rank[i] == hi) b = qt_value(key[i]);
  }
  return qt_lerp(a, b, g);
}

}  // namespace
