// Moulin hydrographs (shakti_set_moulins): the piecewise-linear lookup shared by the device kernel and the host
// (shakti_moulin_discharge, the water budget), so that both give the same bits for the same t.
#pragma once
#include <cmath>
#include <cstdint>

#include <cuda_runtime.h>

namespace shakti {

// Q(t) of one hydrograph with knots (tk[j], qk[j]), j < n, tk strictly increasing: linear between knots, constant
// outside them.  period > 0 first wraps t into [tk[0], tk[0] + period).  Both builds round every operation
// separately (no fused multiply-add), so host and device results are bitwise equal.
__host__ __device__ inline double hydrograph_at(const double* tk, const double* qk, int64_t n, double period, double t) {
  if (period > 0) {
    double r = fmod(t - tk[0], period);   // exact; sign of t - tk[0]
    if (r < 0) r += period;
    t = tk[0] + r;
  }
  if (!(t > tk[0])) return qk[0];
  if (t >= tk[n - 1]) return qk[n - 1];
  int64_t lo = 0, hi = n - 1;             // tk[lo] < t < tk[hi]
  while (hi - lo > 1) {
    const int64_t mid = lo + (hi - lo) / 2;
    if (tk[mid] <= t) lo = mid; else hi = mid;
  }
#ifdef __CUDA_ARCH__
  const double slope = __ddiv_rn(__dsub_rn(qk[hi], qk[lo]), __dsub_rn(tk[hi], tk[lo]));
  return __dadd_rn(__dmul_rn(slope, __dsub_rn(t, tk[lo])), qk[lo]);
#else
  const double slope = (qk[hi] - qk[lo]) / (tk[hi] - tk[lo]);
  volatile double d = slope * (t - tk[lo]);   // volatile: keeps a host compiler from fusing this into an FMA
  return d + qk[lo];
#endif
}

}  // namespace shakti
