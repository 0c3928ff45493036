// Row product of the one-thread-per-row SELL-32 kernels (spmv_sell_kernel, restrict_cheby_first_kernel in
// kernels.cu; amg_cheby_kernel, amg_cheby_h_kernel, amg_resid_h_kernel in amg.cu).
#pragma once
#include <cuda_fp16.h>

#include <cstdint>
#include <type_traits>

namespace shakti {

// Row bound RB of sell_row_product for a matrix with values of type V and longest row max_width
// (DevSell::max_width).  Measured at C4 on a B200 (1000 W): with rows of <= 8 entries the fp32 kernels gain
// 10-25 % (fine-level smoother 271 -> 216 us); a bound of 32 on the rows of 21-28 entries of the restriction and
// of level 1 made those kernels three times slower (80 registers), and the fp64 Krylov SpMV lost 14 % at bound 8
// (48 registers).  The opt-in half-precision copy has not been timed at bound 8 (38 instead of 26-28 registers).
// So only fp32 matrices with rows of <= 8 entries take RB = 8; everything else keeps the plain loop (RB = 0).
template <class V, class F>
inline void sell_row_bound_dispatch(int32_t max_width, F&& launch) {
  if constexpr (std::is_same_v<V, float>) {
    if (max_width <= 8) return launch(std::integral_constant<int, 8>{});
  }
  launch(std::integral_constant<int, 0>{});
}

#ifdef __CUDACC__
__device__ __forceinline__ float sell_entry(__half v) { return __half2float(v); }
__device__ __forceinline__ float sell_entry(float v) { return v; }
__device__ __forceinline__ double sell_entry(double v) { return v; }

// sum_k val[k] x[col[k]] over the w entries of one row (cp, vp: the row's entry 0; entry k is 32 further on),
// accumulated k = 0 ... w-1 into one accumulator, one FMA per entry.  The loads are latency bound: with
// RB > 0 (w <= RB) the row's columns and values are all loaded first, then all its gathers are issued,
// and only then does the FMA chain start, so a thread has the whole row in flight instead of the few
// entries an unrolled loop overlaps.  RB = 0: plain loop.
template <int RB, class T, class V>
__device__ __forceinline__ T sell_row_product(const int32_t* __restrict__ cp, const V* __restrict__ vp, int32_t w,
                                              const T* __restrict__ x) {
  T acc = 0;
  if constexpr (RB > 0) {
    int32_t c[RB];
    V v[RB];
    T xv[RB];
#pragma unroll
    for (int k = 0; k < RB; ++k)
      if (k < w) {
        c[k] = cp[32 * k];
        v[k] = vp[32 * k];
      }
#pragma unroll
    for (int k = 0; k < RB; ++k)
      if (k < w) xv[k] = x[c[k]];
#pragma unroll
    for (int k = 0; k < RB; ++k)
      if (k < w) acc += sell_entry(v[k]) * xv[k];
  } else {
#pragma unroll 4
    for (int k = 0; k < w; ++k) acc += sell_entry(vp[32 * k]) * x[cp[32 * k]];
  }
  return acc;
}
#endif

}  // namespace shakti
