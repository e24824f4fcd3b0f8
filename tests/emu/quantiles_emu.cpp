// quantiles_emu.cpp - host lock-step build of trpl_fit_quantiles: the selection routines the CUDA
// kernel runs (metrotrpl_b200/csrc/fit_quantiles.h) compiled with g++, with the histograms of every
// radix pass built by a loop over the column instead of shared-memory atomics.  Test infrastructure
// only, built and loaded by tests/emu/quantiles_emu.py; never reachable from the metrotrpl_b200 package.
#define TRPL_HOST_EMU 1
#include <stdint.h>
#include <algorithm>
#include <vector>
#include "../../metrotrpl_b200/csrc/fit_quantiles.h"

// The library's trpl_fit_quantiles on a host fit buffer [n_sets][n_cols]: the radix select of
// fit_quantiles.h, with the histograms of every pass built by a loop over the column.  Returns null, or
// the message the call is refused with.
extern "C" const char* trpl_emu_fit_quantiles(int32_t n_sets, int32_t n_cols, const double* fit, int32_t n_q,
                                              const double* q, double* quant, int32_t* count) {
  if (const char* why = qt_check(n_q, q)) return why;
#pragma omp parallel for schedule(dynamic, 16)
  for (int k = 0; k < n_cols; ++k) {
    std::vector<uint64_t> keys;
    for (int s = 0; s < n_sets; ++s) {
      const double x = fit[(size_t)s * n_cols + k];
      if (!isnan(x)) keys.push_back(qt_key(x));
    }
    const int n = (int)keys.size();
    int rank[QT_MAX_TARGETS];
    uint32_t left[QT_MAX_TARGETS];
    uint64_t pre[QT_MAX_TARGETS] = {};
    const int nt = qt_targets(n, n_q, q, rank);
    for (int t = 0; t < nt; ++t) left[t] = (uint32_t)rank[t];
    std::vector<uint32_t> hist(QT_BINS);
    for (int p = 0; p < QT_PASSES; ++p) {
      uint64_t next[QT_MAX_TARGETS];
      for (int t = 0; t < nt; ++t) {
        std::fill(hist.begin(), hist.end(), 0u);
        for (uint64_t key : keys)
          if (qt_match(key, pre[t], p)) ++hist[(key >> qt_shift(p)) & (QT_BINS - 1)];
        next[t] = pre[t] | (uint64_t)qt_pick(hist.data(), left[t]) << qt_shift(p);
      }
      for (int t = 0; t < nt; ++t) pre[t] = next[t];
    }
    for (int j = 0; j < n_q; ++j) quant[(size_t)j * n_cols + k] = qt_finish(n, q[j], rank, pre, nt);
    if (count) count[k] = n;
  }
  return nullptr;
}
