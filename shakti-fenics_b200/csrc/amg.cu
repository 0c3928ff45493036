// Smoothed-aggregation AMG (see amg.h).  Symbolic phase on the host (patterns are fixed by
// the mesh), numeric phase and V-cycle on the device.
#include "amg.h"
#include "comm.h"

#include <algorithm>
#include <cstdlib>
#include <cmath>
#include <map>
#include <numeric>

namespace shakti {

// ------------------------------------------------------------------ host: aggregation + patterns

// Greedy (Vanek) aggregation on the graph of STRONG connections of the square block of A
// (strong[k] != 0 for CSR entry k; empty = every connection is strong).
// Returns agg[i] in [0,n_agg) or -1 for excluded rows.
static int aggregate(const HostCsr& A, int32_t n, const std::vector<uint8_t>& excl, const std::vector<uint8_t>& strong,
                     std::vector<int32_t>& agg) {
  agg.assign(n, -1);
  std::vector<uint8_t> free_(n, 1);
  for (int32_t i = 0; i < n; ++i)
    if (!excl.empty() && excl[i]) free_[i] = 0;
  int32_t na = 0;
  auto nb = [&](int32_t i, auto&& f) {
    for (int32_t k = A.rowptr[i]; k < A.rowptr[i + 1]; ++k) {
      const int32_t j = A.col[k];
      if (j < n && j != i && (excl.empty() || !excl[j]) && (strong.empty() || strong[k])) f(j);
    }
  };
  // pass 1: roots whose whole neighbourhood is free
  for (int32_t i = 0; i < n; ++i) {
    if (!free_[i]) continue;
    bool ok = true;
    nb(i, [&](int32_t j) { ok &= (free_[j] != 0); });
    if (!ok) continue;
    agg[i] = na;
    free_[i] = 0;
    nb(i, [&](int32_t j) { agg[j] = na; free_[j] = 0; });
    ++na;
  }
  // pass 2: attach leftovers to a neighbouring pass-1 aggregate (smallest so far)
  {
    std::vector<int32_t> snap(agg);
    std::vector<int32_t> size(na, 0);
    for (int32_t i = 0; i < n; ++i)
      if (snap[i] >= 0) size[snap[i]]++;
    for (int32_t i = 0; i < n; ++i) {
      if (!free_[i]) continue;
      int32_t best = -1;
      nb(i, [&](int32_t j) {
        if (snap[j] >= 0 && (best < 0 || size[snap[j]] < size[best])) best = snap[j];
      });
      if (best >= 0) { agg[i] = best; size[best]++; free_[i] = 0; }
    }
  }
  // pass 3: whatever is left forms aggregates with its free neighbours
  for (int32_t i = 0; i < n; ++i) {
    if (!free_[i]) continue;
    agg[i] = na;
    free_[i] = 0;
    nb(i, [&](int32_t j) { if (free_[j]) { agg[j] = na; free_[j] = 0; } });
    ++na;
  }
  return na;
}

// pattern of A(:, 0:B.n_rows) * B
static HostCsr product_pattern(const HostCsr& A, const HostCsr& B) {
  HostCsr C;
  C.n_rows = A.n_rows;
  C.n_cols = B.n_cols;
  C.rowptr.assign(A.n_rows + 1, 0);
  std::vector<int32_t> mark(B.n_cols, -1), tmp;
  for (int64_t i = 0; i < A.n_rows; ++i) {
    tmp.clear();
    for (int32_t k = A.rowptr[i]; k < A.rowptr[i + 1]; ++k) {
      const int32_t j = A.col[k];
      if (j >= B.n_rows) continue;
      for (int32_t l = B.rowptr[j]; l < B.rowptr[j + 1]; ++l) {
        const int32_t c = B.col[l];
        if (mark[c] != (int32_t)i) { mark[c] = (int32_t)i; tmp.push_back(c); }
      }
    }
    std::sort(tmp.begin(), tmp.end());
    C.col.insert(C.col.end(), tmp.begin(), tmp.end());
    if (C.col.size() > 2000000000ULL) throw Error(SHAKTI_ERR_INVALID, "AMG product pattern too large");
    C.rowptr[i + 1] = (int32_t)C.col.size();
  }
  return C;
}

// ------------------------------------------------------------------ device kernels

// dinv = 1/diag
__global__ void amg_dinv_kernel(int32_t n, const int32_t* __restrict__ diag_pos, const double* __restrict__ val,
                                double* __restrict__ dinv) {
  const int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double d = val[diag_pos[i]];
  dinv[i] = d != 0.0 ? 1.0 / d : 0.0;
}

// P = (I - omega D^-1 A) T : every A entry (i,j) adds (delta_ij - omega a_ij / a_ii) to
// P[i, agg(j)]; pmap holds the position of agg(j) inside P's row i (255: dropped).
__global__ void __launch_bounds__(256)
amg_prolongator_kernel(SellView A, const uint8_t* __restrict__ pmap, const int32_t* __restrict__ diag_pos,
                       const double* __restrict__ dinv, double omega, const int32_t* __restrict__ Pslice,
                       double* __restrict__ Pval) {
  const int32_t row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= A.n_rows) return;
  const int32_t slice = row >> 5, lane = row & 31;
  const int32_t base = A.slice_ptr[slice];
  const int32_t w = (A.slice_ptr[slice + 1] - base) >> 5;
  const int32_t pbase = Pslice[slice] + lane;
  const int32_t dpos = diag_pos[row];
  const double s = omega * dinv[row];
  for (int k = 0; k < w; ++k) {
    const int32_t p = base + 32 * k + lane;
    const uint8_t t = pmap[p];
    if (t == 255) continue;
    const double v = (p == dpos ? 1.0 : 0.0) - s * A.val[p];
    Pval[pbase + 32 * (int32_t)t] += v;
  }
}

// out[p] = src[map[p]] (map < 0 -> 0)
__global__ void amg_gather_vals_kernel(int64_t n, const int32_t* __restrict__ map, const double* __restrict__ src,
                                       double* __restrict__ out) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const int32_t m = map[i];
    out[i] = m >= 0 ? src[m] : 0.0;
  }
}

// C = A(:, 0:B.n_rows) * B with a known pattern of C (values zeroed beforehand): one thread
// per row, positions found by binary search in C's sorted row.
__global__ void __launch_bounds__(128)
amg_spgemm_kernel(SellView A, const int32_t* __restrict__ Alen, SellView B, const int32_t* __restrict__ Blen,
                  int32_t Bn_rows, const int32_t* __restrict__ Cslice, const int32_t* __restrict__ Ccol,
                  const int32_t* __restrict__ Clen, double* __restrict__ Cval) {
  const int32_t row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= A.n_rows) return;
  const int32_t lane = row & 31;
  const int32_t abase = A.slice_ptr[row >> 5] + lane;
  const int32_t cbase = Cslice[row >> 5] + lane;
  const int32_t clen = Clen[row];
  const int32_t alen = Alen[row];
  for (int ka = 0; ka < alen; ++ka) {
    const int32_t j = A.col[abase + 32 * ka];
    if (j >= Bn_rows) continue;
    const double a = A.val[abase + 32 * ka];
    if (a == 0.0) continue;
    const int32_t bbase = B.slice_ptr[j >> 5] + (j & 31);
    const int32_t blen = Blen[j];
    for (int kb = 0; kb < blen; ++kb) {
      const int32_t c = B.col[bbase + 32 * kb];
      const double b = B.val[bbase + 32 * kb];
      int lo = 0, hi = clen - 1;
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (Ccol[cbase + 32 * mid] < c) lo = mid + 1; else hi = mid;
      }
      Cval[cbase + 32 * lo] += a * b;
    }
  }
}

// Same product with one WARP per row, for the small levels where one thread per row leaves the GPU
// idle and the rows of R are long: each lane owns output positions of C's row (lane, lane+32, ...)
// and accumulates its entries itself -> no atomics, same summation order every run.
__global__ void __launch_bounds__(128)
amg_spgemm_warp_kernel(SellView A, const int32_t* __restrict__ Alen, SellView B, const int32_t* __restrict__ Blen,
                       int32_t Bn_rows, const int32_t* __restrict__ Cslice, const int32_t* __restrict__ Ccol,
                       const int32_t* __restrict__ Clen, double* __restrict__ Cval) {
  const int32_t row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= A.n_rows) return;
  const int32_t abase = A.slice_ptr[row >> 5] + (row & 31);
  const int32_t cbase = Cslice[row >> 5] + (row & 31);
  const int32_t clen = Clen[row], alen = Alen[row];
  for (int pos = lane; pos < clen; pos += 32) {
    const int32_t c = Ccol[cbase + 32 * pos];
    double acc = 0.0;
    for (int ka = 0; ka < alen; ++ka) {
      const int32_t j = A.col[abase + 32 * ka];
      if (j >= Bn_rows) continue;
      const double a = A.val[abase + 32 * ka];
      if (a == 0.0) continue;
      const int32_t bbase = B.slice_ptr[j >> 5] + (j & 31);
      int lo = 0, hi = Blen[j] - 1;
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (B.col[bbase + 32 * mid] < c) lo = mid + 1; else hi = mid;
      }
      if (hi >= 0 && lo == hi && B.col[bbase + 32 * lo] == c) acc += a * B.val[bbase + 32 * lo];
    }
    Cval[cbase + 32 * pos] = acc;
  }
}

// ---- table-driven product for the large levels.  The patterns are fixed by the mesh, so the position of
// every product a_ik b_kj inside C's row is found ONCE (the binary search above, run by
// amg_spgemm_slots_kernel) and kept as one byte per product, stored slice-interleaved like the matrices:
// product t of row r at prod_ptr[r >> 5] + 32 t + (r & 31).  The numeric product then streams A, the
// table and the gathered rows of B, accumulates C's row in shared memory (no global read-modify-write,
// no search) and writes it once.
struct SpgemmPlan {
  bool built = false, ok = false;
  DevBuf<int64_t> prod_ptr;   // n_slices + 1
  DevBuf<uint8_t> slot;
};

// per slice: 32 x (largest number of products of any of its rows)
__global__ void __launch_bounds__(128)
amg_spgemm_count_kernel(SellView A, const int32_t* __restrict__ Alen, const int32_t* __restrict__ Blen, int32_t Bn_rows,
                        int32_t* __restrict__ slice_width) {
  const int32_t row = blockIdx.x * blockDim.x + threadIdx.x;
  int32_t cnt = 0;
  if (row < A.n_rows) {
    const int32_t abase = A.slice_ptr[row >> 5] + (row & 31);
    const int32_t alen = Alen[row];
    for (int ka = 0; ka < alen; ++ka) {
      const int32_t j = A.col[abase + 32 * ka];
      if (j < Bn_rows) cnt += Blen[j];
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) cnt = max(cnt, __shfl_xor_sync(0xffffffffu, cnt, o));
  if ((threadIdx.x & 31) == 0 && (row >> 5) < A.n_slices) slice_width[row >> 5] = cnt;
}

__global__ void __launch_bounds__(128)
amg_spgemm_slots_kernel(SellView A, const int32_t* __restrict__ Alen, SellView B, const int32_t* __restrict__ Blen,
                        int32_t Bn_rows, const int32_t* __restrict__ Cslice, const int32_t* __restrict__ Ccol,
                        const int32_t* __restrict__ Clen, const int64_t* __restrict__ prod_ptr, uint8_t* __restrict__ slot) {
  const int32_t row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= A.n_rows) return;
  const int32_t lane = row & 31;
  const int32_t abase = A.slice_ptr[row >> 5] + lane;
  const int32_t cbase = Cslice[row >> 5] + lane;
  const int32_t clen = Clen[row], alen = Alen[row];
  uint8_t* __restrict__ sp = slot + prod_ptr[row >> 5] + lane;
  int64_t t = 0;
  for (int ka = 0; ka < alen; ++ka) {
    const int32_t j = A.col[abase + 32 * ka];
    if (j >= Bn_rows) continue;
    const int32_t bbase = B.slice_ptr[j >> 5] + (j & 31);
    const int32_t blen = Blen[j];
    for (int kb = 0; kb < blen; ++kb, ++t) {
      const int32_t c = B.col[bbase + 32 * kb];
      int lo = 0, hi = clen - 1;
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (Ccol[cbase + 32 * mid] < c) lo = mid + 1; else hi = mid;
      }
      sp[32 * t] = (uint8_t)lo;
    }
  }
}

__global__ void __launch_bounds__(128)
amg_spgemm_table_kernel(SellView A, const int32_t* __restrict__ Alen, SellView B, const int32_t* __restrict__ Blen,
                        int32_t Bn_rows, const int32_t* __restrict__ Cslice, const int32_t* __restrict__ Clen,
                        const int64_t* __restrict__ prod_ptr, const uint8_t* __restrict__ slot, double* __restrict__ Cval) {
  extern __shared__ double acc[];   // [C width][128]: entry k of this thread's row at acc[k * 128 + threadIdx.x]
  const int32_t row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= A.n_rows) return;
  const int32_t lane = row & 31;
  const int32_t abase = A.slice_ptr[row >> 5] + lane;
  const int32_t clen = Clen[row], alen = Alen[row];
  double* __restrict__ my = acc + threadIdx.x;
  for (int k = 0; k < clen; ++k) my[k * 128] = 0.0;
  const uint8_t* __restrict__ sp = slot + prod_ptr[row >> 5] + lane;
  int64_t t = 0;
  for (int ka = 0; ka < alen; ++ka) {
    const int32_t j = A.col[abase + 32 * ka];
    if (j >= Bn_rows) continue;
    const double a = A.val[abase + 32 * ka];
    const int32_t bbase = B.slice_ptr[j >> 5] + (j & 31);
    const int32_t blen = Blen[j];
    for (int kb = 0; kb < blen; ++kb, ++t) my[(int)sp[32 * t] * 128] += a * B.val[bbase + 32 * kb];
  }
  double* __restrict__ cp = Cval + Cslice[row >> 5] + lane;
  for (int k = 0; k < clen; ++k) cp[32 * k] = my[k * 128];
}

static void build_spgemm_plan(const DevSell& A, const DevSell& B, const DevSell& C, SpgemmPlan& plan, cudaStream_t s) {
  plan.built = true;
  plan.ok = false;
  const size_t smem = (size_t)C.max_width * 128 * sizeof(double);
  if (A.n_rows == 0 || C.max_width > 255 || smem > 96 * 1024) return;
  DevBuf<int32_t> width;
  width.alloc_zero(A.n_slices, s);
  SHAKTI_LAUNCH(amg_spgemm_count_kernel, div_up((int64_t)A.n_slices * 32, 128), 128, 0, s, view(A), A.rowlen.p, B.rowlen.p, B.n_rows,
                width.p);
  const std::vector<int32_t> w = width.download(s);
  std::vector<int64_t> ptr(w.size() + 1, 0);
  for (size_t i = 0; i < w.size(); ++i) ptr[i + 1] = ptr[i] + 32 * (int64_t)w[i];
  plan.prod_ptr.upload(ptr);
  plan.slot.alloc((size_t)std::max<int64_t>(ptr.back(), 1));
  SHAKTI_LAUNCH(amg_spgemm_slots_kernel, div_up(A.n_rows, 128), 128, 0, s, view(A), A.rowlen.p, view(B), B.rowlen.p, B.n_rows,
                C.slice_ptr.p, C.col.p, C.rowlen.p, plan.prod_ptr.p, plan.slot.p);
  if (smem > 48 * 1024)
    SHAKTI_CUDA(cudaFuncSetAttribute(amg_spgemm_table_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
  plan.ok = true;
}

// C = A B numerically (pattern of C known): table-driven thread-per-row for large matrices, warp-per-row for small ones
static void spgemm_numeric(const DevSell& A, const DevSell& B, DevSell& C, SpgemmPlan& plan, cudaStream_t s) {
  if (A.n_rows == 0) return;
  if (A.n_rows <= 400000) {
    SHAKTI_LAUNCH(amg_spgemm_warp_kernel, div_up((int64_t)A.n_rows * 32, 128), 128, 0, s, view(A), A.rowlen.p, view(B), B.rowlen.p,
                  B.n_rows, C.slice_ptr.p, C.col.p, C.rowlen.p, C.val.p);
    return;
  }
  if (!plan.built) build_spgemm_plan(A, B, C, plan, s);
  if (plan.ok) {
    SHAKTI_LAUNCH(amg_spgemm_table_kernel, div_up(A.n_rows, 128), 128, (size_t)C.max_width * 128 * sizeof(double), s, view(A),
                  A.rowlen.p, view(B), B.rowlen.p, B.n_rows, C.slice_ptr.p, C.rowlen.p, plan.prod_ptr.p, plan.slot.p, C.val.p);
  } else {
    SHAKTI_CUDA(cudaMemsetAsync(C.val.p, 0, sizeof(double) * C.padded, s));
    SHAKTI_LAUNCH(amg_spgemm_kernel, div_up(A.n_rows, 128), 128, 0, s, view(A), A.rowlen.p, view(B), B.rowlen.p, B.n_rows,
                  C.slice_ptr.p, C.col.p, C.rowlen.p, C.val.p);
  }
}

// dense coarse operator: D[i*ld + j] (ld = 2n), right half = identity
__global__ void amg_dense_fill_kernel(SellView A, const int32_t* __restrict__ Alen, int32_t n, double* __restrict__ D) {
  const int32_t row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= n) return;
  const int32_t base = A.slice_ptr[row >> 5] + (row & 31);
  for (int k = 0; k < Alen[row]; ++k) {
    const int32_t j = A.col[base + 32 * k];
    if (j < n) D[(size_t)row * 2 * n + j] += A.val[base + 32 * k];
  }
  D[(size_t)row * 2 * n + n + row] = 1.0;
}

// Gauss-Jordan with partial pivoting on [A | I] -> [I | A^-1], one thread block.
__global__ void __launch_bounds__(1024)
amg_dense_invert_kernel(int32_t n, double* __restrict__ D, int* __restrict__ info) {
  extern __shared__ double fcol[];   // n factors
  __shared__ int piv;
  __shared__ double pval;
  const int ld = 2 * n;
  for (int k = 0; k < n; ++k) {
    if (threadIdx.x < 32) {   // warp-parallel pivot search (first maximum wins)
      int p = k;
      double best = -1.0;
      for (int i = k + (int)threadIdx.x; i < n; i += 32) {
        const double v = fabs(D[(size_t)i * ld + k]);
        if (v > best) { best = v; p = i; }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const double ob = __shfl_xor_sync(0xffffffffu, best, o);
        const int op = __shfl_xor_sync(0xffffffffu, p, o);
        if (ob > best || (ob == best && op < p)) { best = ob; p = op; }
      }
      if (threadIdx.x == 0) {
        piv = p;
        pval = D[(size_t)p * ld + k];
        if (!(best > 0.0)) *info = k + 1;
      }
    }
    __syncthreads();
    const int p = piv;
    const double inv = pval != 0.0 ? 1.0 / pval : 0.0;
    // swap rows k,p and scale the pivot row
    for (int j = threadIdx.x; j < ld; j += blockDim.x) {
      const double a = D[(size_t)p * ld + j], b = D[(size_t)k * ld + j];
      D[(size_t)p * ld + j] = b;
      D[(size_t)k * ld + j] = a * inv;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += blockDim.x) fcol[i] = (i == k) ? 0.0 : D[(size_t)i * ld + k];
    __syncthreads();
    for (int idx = threadIdx.x; idx < n * ld; idx += blockDim.x) {
      const int i = idx / ld, j = idx - i * ld;
      const double f = fcol[i];
      if (f != 0.0) D[(size_t)i * ld + j] -= f * D[(size_t)k * ld + j];
    }
    __syncthreads();
  }
}

// x = Ainv b, Ainv = right half of D; one warp per row
template <class TB, class TX>
__global__ void amg_dense_apply_kernel(int32_t n, const double* __restrict__ D, const TB* __restrict__ b,
                                       TX* __restrict__ x) {
  pdl_sync();
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= n) return;
  const double* row = D + (size_t)warp * 2 * n + n;
  double acc = 0.0;
  for (int j = lane; j < n; j += 32) acc += row[j] * (double)b[j];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) x[warp] = (TX)acc;
}

// ------------------------------------------------------------------ smoother kernels
// Chebyshev step: r = dinv (b - A x); d = c1 d + c2 r; x_out = x + d
// KG as in spmv_sell_kernel (kernels.cu): 1 = thread per row, 8 = block per slice for small wide-rowed levels.
// RB (KG = 1): row bound of sell_row_product (sell_row.h), picked by sell_row_bound_dispatch from the longest row.
// cf = {c1, c2} in device memory (amg_cheby_coef_kernel), so that a new spectral bound changes no kernel argument.
// MODE, for the fine level of the mixed-precision cycle (Amg::apply):
//   CHEBY_X_IS_D  first sweep after amg_cycle_entry_kernel, which wrote the first iterate to x only: the old d is x
//   CHEBY_EXIT    last sweep of the cycle: z = (double)(x + d_new); d is read, d and x_out are not written
enum { CHEBY_PLAIN = 0, CHEBY_X_IS_D = 1, CHEBY_EXIT = 2 };
template <class T, int KG, int MODE = CHEBY_PLAIN, int RB = 0>
__global__ void __launch_bounds__(256)
amg_cheby_kernel(SellViewT<T> A, const T* __restrict__ dinv, const T* __restrict__ b, const T* __restrict__ x,
                 T* __restrict__ d, T* __restrict__ x_out, const double* __restrict__ cf, double* __restrict__ z) {
  pdl_sync();
  int32_t row;
  T acc = 0;
  if (KG == 1) {
    row = blockIdx.x * blockDim.x + threadIdx.x;
    const int32_t slice = row >> 5;
    if (slice >= A.n_slices) return;
    const int32_t base = A.slice_ptr[slice];
    const int32_t w = (A.slice_ptr[slice + 1] - base) >> 5;
    acc = sell_row_product<RB>(A.col + base + (row & 31), A.val + base + (row & 31), w, x);
  } else {
    __shared__ T psum[KG][32];
    const int32_t slice = blockIdx.x;
    const int lane = threadIdx.x & 31, g = threadIdx.x >> 5;
    row = slice * 32 + lane;
    const int32_t base = A.slice_ptr[slice];
    const int32_t w = (A.slice_ptr[slice + 1] - base) >> 5;
    const int32_t* __restrict__ cp = A.col + base + lane;
    const T* __restrict__ vp = A.val + base + lane;
    for (int k = g; k < w; k += KG) acc += vp[32 * k] * x[cp[32 * k]];
    psum[g][lane] = acc;
    __syncthreads();
    if (g != 0) return;
#pragma unroll
    for (int j = 1; j < KG; ++j) acc += psum[j][lane];
  }
  if (row >= A.n_rows) return;
  const T c1 = (T)cf[0], c2 = (T)cf[1];
  const T r = dinv[row] * (b[row] - acc);
  const T dn = c1 * (MODE == CHEBY_X_IS_D ? x[row] : d[row]) + c2 * r;
  if (MODE == CHEBY_EXIT) {
    z[row] = (double)(x[row] + dn);
    return;
  }
  d[row] = dn;
  x_out[row] = x[row] + dn;
}
constexpr int32_t kChebyWideRowsBelow = 300000;
template <class T, int MODE = CHEBY_PLAIN>
static void launch_cheby(SellViewT<T> A, const T* dinv, const T* b, const T* x, T* d, T* x_out, const double* cf, cudaStream_t s) {
  static_assert(MODE != CHEBY_EXIT, "the exit sweep writes z: launched by Amg::apply");
  // (a variant interleaving two slices per warp was measured slower: 193 vs 179 ms per step)
  if (A.n_rows < kChebyWideRowsBelow)
    SHAKTI_LAUNCH_PDL((amg_cheby_kernel<T, 8, MODE>), A.n_slices, 256, 0, s, A, dinv, b, x, d, x_out, cf, nullptr);
  else
    sell_row_bound_dispatch<T>(A.max_width, [&](auto rb) {
      SHAKTI_LAUNCH_PDL((amg_cheby_kernel<T, 1, MODE, rb.value>), div_up((int64_t)A.n_slices * 32, 256), 256, 0, s, A, dinv, b, x, d,
                        x_out, cf, nullptr);
    });
}

// ---- the same two kernels of the LARGE levels on the half-precision, row-scaled copy Ah = D^-1 A (unit
// diagonal): 6 instead of 8 bytes per stored entry on kernels that are purely bandwidth bound.  The vectors
// stay fp32 and the products are accumulated in fp32; the 5e-4 relative rounding of the entries perturbs the
// PRECONDITIONER only (the Krylov operator and the Galerkin products use the fp64 values).
//   Chebyshev step:  r = dinv b - Ah x ;  d = c1 d + c2 r ;  x_out = x + d
__global__ void __launch_bounds__(256)
amg_cheby_h_kernel(int32_t n_rows, int32_t n_slices, const int32_t* __restrict__ slice_ptr, const int32_t* __restrict__ col,
                   const __half* __restrict__ val, const float* __restrict__ dinv, const float* __restrict__ b,
                   const float* __restrict__ x, float* __restrict__ d, float* __restrict__ x_out, const double* __restrict__ cf) {
  pdl_sync();
  const int32_t row = blockIdx.x * blockDim.x + threadIdx.x;
  const int32_t slice = row >> 5;
  if (slice >= n_slices) return;
  const int32_t base = slice_ptr[slice];
  const int32_t w = (slice_ptr[slice + 1] - base) >> 5;
  const float acc = sell_row_product<0>(col + base + (row & 31), val + base + (row & 31), w, x);
  if (row >= n_rows) return;
  const float c1 = (float)cf[0], c2 = (float)cf[1];
  const float r = dinv[row] * b[row] - acc;
  const float dn = c1 * d[row] + c2 * r;
  d[row] = dn;
  x_out[row] = x[row] + dn;
}
//   residual:  r = b - A x = b - (Ah x) / dinv
__global__ void __launch_bounds__(256)
amg_resid_h_kernel(int32_t n_rows, int32_t n_slices, const int32_t* __restrict__ slice_ptr, const int32_t* __restrict__ col,
                   const __half* __restrict__ val, const float* __restrict__ dinv, const float* __restrict__ b,
                   const float* __restrict__ x, float* __restrict__ r) {
  pdl_sync();
  const int32_t row = blockIdx.x * blockDim.x + threadIdx.x;
  const int32_t slice = row >> 5;
  if (slice >= n_slices) return;
  const int32_t base = slice_ptr[slice];
  const int32_t w = (slice_ptr[slice + 1] - base) >> 5;
  const float acc = sell_row_product<0>(col + base + (row & 31), val + base + (row & 31), w, x);
  if (row >= n_rows) return;
  const float di = dinv[row];
  r[row] = b[row] - (di != 0.f ? acc / di : 0.f);
}
// does level operator A run on its half-precision copy?
static bool uses_half(const Amg::Impl& I, const DevSell& A);

// V-cycle entry on the fine level of the mixed-precision cycle: b = (float)r, and the first Chebyshev step from a
// zero guess, x = (dinv b)/theta -- the work of d2f_kernel and amg_cheby_first_kernel in one pass.  d is not
// written: the next sweep reads x in its place (CHEBY_X_IS_D).
__global__ void amg_cycle_entry_kernel(int32_t n, const double* __restrict__ r, const float* __restrict__ dinv,
                                       const double* __restrict__ inv_theta, float* __restrict__ b, float* __restrict__ x) {
  const int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float bi = (float)r[i];
  b[i] = bi;
  x[i] = dinv[i] * bi * (float)inv_theta[0];
}

// first Chebyshev step from a zero guess: d = (dinv b)/theta ; x = d   (inv_theta = 1/theta in device memory)
template <class T>
__global__ void amg_cheby_first_kernel(int32_t n, const T* __restrict__ dinv, const T* __restrict__ b,
                                       const double* __restrict__ inv_theta, T* __restrict__ d, T* __restrict__ x) {
  pdl_sync();
  const int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const T v = dinv[i] * b[i] * (T)inv_theta[0];
  d[i] = v;
  x[i] = v;
}

// Block maximum of v (256 threads), then one integer atomicMax on the bit pattern (valid for non-negative
// doubles).  A maximum does not depend on the order of its operands, so the result is the same bits however the
// rows are split among threads and blocks.
__device__ __forceinline__ void block_max_to(double v, unsigned long long* __restrict__ out) {
  __shared__ double wmax[8];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  if ((threadIdx.x & 31) == 0) wmax[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x == 0) {
#pragma unroll
    for (int j = 1; j < 8; ++j) v = fmax(v, wmax[j]);
    if (v > 0.0) atomicMax(out, (unsigned long long)__double_as_longlong(v));
  }
}
// few blocks with a grid-stride loop: one same-address atomic per block (one per warp, 500 000 at 16M rows, took
// four times as long as streaming the matrix)
static int bound_blocks(int64_t rows, int sm_count) { return (int)std::min<int64_t>((int64_t)sm_count * 8, std::max<int64_t>(1, div_up(rows, 256))); }

// Gershgorin bound of lambda_max(D^-1 A): max_i |dinv_i| sum_j |a_ij|
__global__ void __launch_bounds__(256)
amg_gershgorin_kernel(SellView A, const double* __restrict__ dinv, unsigned long long* __restrict__ out) {
  double v = 0.0;
  for (int32_t row = blockIdx.x * blockDim.x + threadIdx.x; row < A.n_rows; row += gridDim.x * blockDim.x) {
    const int32_t base = A.slice_ptr[row >> 5] + (row & 31);
    const int32_t w = (A.slice_ptr[(row >> 5) + 1] - A.slice_ptr[row >> 5]) >> 5;
    double acc = 0.0;
    for (int k = 0; k < w; ++k) acc += fabs(A.val[base + 32 * k]);
    v = fmax(v, fabs(dinv[row]) * acc);
  }
  block_max_to(v, out);
}

// The fine level's smoother refresh in one pass over its fp64 values (mixed-precision cycle, Chebyshev smoother).
// Per row: the diagonal, picked out by its slot; dinv in fp64 and fp32; the fp32 copy of every stored entry,
// padding slots and the padding rows of the last slice included (F32 = false: the level runs on its half-precision
// copy, made afterwards from dinv); and the row's Gershgorin number |dinv_i| sum_j |a_ij|.  Same operations in the
// same order as amg_dinv_kernel, d2f_kernel and amg_gershgorin_kernel, so the results are the same bits.
template <bool F32>
__global__ void __launch_bounds__(256)
amg_fine_refresh_kernel(SellView A, const int32_t* __restrict__ diag_pos, double* __restrict__ dinv, float* __restrict__ dinvf,
                        float* __restrict__ valf, unsigned long long* __restrict__ bound) {
  double v = 0.0;
  const int32_t rows = A.n_slices * 32;
  for (int32_t row = blockIdx.x * blockDim.x + threadIdx.x; row < rows; row += gridDim.x * blockDim.x) {
    const int32_t base = A.slice_ptr[row >> 5] + (row & 31);
    const int32_t w = (A.slice_ptr[(row >> 5) + 1] - A.slice_ptr[row >> 5]) >> 5;
    double di = 0.0;
    if (row < A.n_rows) {
      const double d = A.val[diag_pos[row]];
      di = d != 0.0 ? 1.0 / d : 0.0;
      dinv[row] = di;
      dinvf[row] = (float)di;
    }
    double acc = 0.0;
#pragma unroll 4
    for (int k = 0; k < w; ++k) {
      const double a = A.val[base + 32 * k];
      if (F32) valf[base + 32 * k] = (float)a;
      acc += fabs(a);
    }
    if (row < A.n_rows) v = fmax(v, fabs(di) * acc);
  }
  block_max_to(v, bound);
}

// Chebyshev coefficients of levels [0, nl) from their bounds of lambda_max(D^-1 A), kept in device memory so that a
// new bound needs no host round trip and changes no kernel argument of the captured V-cycle.  Per level (stride
// `stride`): [0] = 1/theta, then sweep k's pair (c1, c2) at [2 + 2k].  A bound that is not positive and finite gives
// 2.0, or with `keep` leaves the level's previous value.  The formulas and the order of the operations are those the
// host used; the _rn intrinsics keep the compiler from contracting any of them into a fused multiply-add.
__global__ void amg_cheby_coef_kernel(int nl, int sweeps, int stride, double ratio, const double* __restrict__ bound, int keep,
                                      double* __restrict__ lmax, double* __restrict__ coef) {
  if (blockIdx.x != 0 || threadIdx.x != 0) return;
  for (int l = 0; l < nl; ++l) {
    const double h = bound[l];
    if (h > 0.0 && isfinite(h)) lmax[l] = h;
    else if (!keep) lmax[l] = 2.0;
    const double hi = lmax[l], lo = __ddiv_rn(hi, ratio);
    const double theta = __dmul_rn(0.5, __dadd_rn(hi, lo)), delta = __dmul_rn(0.5, __dsub_rn(hi, lo));
    const double sigma = __ddiv_rn(theta, delta);
    double rho = __ddiv_rn(1.0, sigma);
    double* __restrict__ c = coef + (size_t)l * stride;
    c[0] = __ddiv_rn(1.0, theta);
    c[2] = 0.0;    // sweep 0 from a nonzero guess
    c[3] = c[0];
    for (int k = 1; k < sweeps; ++k) {
      const double rho_n = __ddiv_rn(1.0, __dsub_rn(__dmul_rn(2.0, sigma), rho));
      c[2 + 2 * k] = __dmul_rn(rho_n, rho);
      c[3 + 2 * k] = __ddiv_rn(__dmul_rn(2.0, rho_n), delta);
      rho = rho_n;
    }
  }
}

// ------------------------------------------------------------------ distributed helpers
// sendbuf[s*w + k] = pos >= 0 ? val[pos] : 0
__global__ void amg_pack_rows_kernel(int64_t n, const int32_t* __restrict__ pos, const double* __restrict__ val,
                                     double* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int32_t p = pos[i];
  out[i] = p >= 0 ? val[p] : 0.0;
}
// val[pos[i]] = in[i] where pos >= 0
__global__ void amg_unpack_rows_kernel(int64_t n, const int32_t* __restrict__ pos, const double* __restrict__ in,
                                       double* __restrict__ val) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int32_t p = pos[i];
  if (p >= 0) val[p] = in[i];
}
// rows of the (distributed) coarsest operator as dense rows in GLOBAL column numbering
__global__ void amg_dense_rows_kernel(SellView A, const int32_t* __restrict__ Alen, const int32_t* __restrict__ colmap,
                                      int32_t n, int32_t N, double* __restrict__ D) {
  const int32_t row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= n) return;
  const int32_t base = A.slice_ptr[row >> 5] + (row & 31);
  for (int k = 0; k < Alen[row]; ++k) D[(size_t)row * N + colmap[A.col[base + 32 * k]]] += A.val[base + 32 * k];
}
// gathered row blocks [rank][nmax][N] -> [A | I] with leading dimension 2N
__global__ void amg_dense_assemble_kernel(int32_t N, int32_t nmax, int32_t nranks, const int32_t* __restrict__ off,
                                          const double* __restrict__ G, double* __restrict__ D) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (int64_t)N * N) return;
  const int32_t gi = (int32_t)(t / N), j = (int32_t)(t - (int64_t)gi * N);
  int r = 0;
  while (r + 1 < nranks && off[r + 1] <= gi) ++r;
  const int32_t li = gi - off[r];
  D[(size_t)gi * 2 * N + j] = G[((size_t)r * nmax + li) * N + j];
  if (j == 0) D[(size_t)gi * 2 * N + N + gi] = 1.0;
}
// gathered rhs blocks [rank][nmax] -> global vector
template <class TO>
__global__ void amg_compact_kernel(int32_t N, int32_t nmax, int32_t nranks, const int32_t* __restrict__ off,
                                   const double* __restrict__ G, TO* __restrict__ out) {
  const int32_t gi = blockIdx.x * blockDim.x + threadIdx.x;
  if (gi >= N) return;
  int r = 0;
  while (r + 1 < nranks && off[r + 1] <= gi) ++r;
  out[gi] = (TO)G[(size_t)r * nmax + (gi - off[r])];
}

// out[i] = src[map[i]]
template <class T>
__global__ void amg_gather_map_kernel(int32_t n, const int32_t* __restrict__ map, const T* __restrict__ src, T* __restrict__ out) {
  pdl_sync();
  const int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = src[map[i]];
}

template <class TI, class TO>
__global__ void amg_convert_kernel(int32_t n, const TI* __restrict__ in, TO* __restrict__ out) {
  const int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = (TO)in[i];
}

// ------------------------------------------------------------------ hierarchy
template <class T>
struct CycleVecs {
  DevBuf<T> x, x2, b, r, d, dinv;
};

struct AmgLevel {
  int32_t n = 0, n_ghost = 0, n_cols = 0;      // owned rows, ghost columns, n + n_ghost
  int32_t n_coarse = 0, n_coarse_ghost = 0;
  int64_t nnz = 0;
  DevSell A;                  // levels >= 1 (level 0 uses the caller's matrix)
  DevBuf<int32_t> diag_pos;   // levels >= 1
  DevBuf<double> dinv;
  DevSell P, R, AP;           // P: (n + n_ghost) x (n_coarse + n_coarse_ghost); R = (P[owned, owned])^T
  SpgemmPlan plan_AP, plan_RAP;
  DevBuf<uint8_t> pmap;
  DevBuf<int32_t> tmap;
  CycleVecs<double> vd;       // V-cycle work vectors, double ...
  CycleVecs<float> vf;        // ... or single precision (mixed-precision cycle)
  int32_t index = 0;          // position in the hierarchy
  bool last = false;
  HostCsr hA;                 // host pattern (levels >= 1)
  HostSell hS;
  // halo of this level's vectors (level 0: the caller's plan)
  std::vector<Neighbor> nbrs;
  HaloPlan own_halo;
  HaloPlan* halo = nullptr;
  // exchange of the prolongator rows of interface vertices
  int maxw = 0;
  DevBuf<int32_t> psend_pos, pg_pos;
  DevBuf<double> psend, precv;
};

struct Amg::Impl {
  AmgOptions opt;
  cudaStream_t s = 0;
  const HostCsr* A0 = nullptr;
  const HostSell* S0 = nullptr;
  const std::vector<Neighbor>* nbrs0 = nullptr;
  HaloPlan* halo0 = nullptr;
  std::vector<uint8_t> exclude;
  std::vector<std::unique_ptr<AmgLevel>> lv;
  // coarsest level: gathered on every rank and inverted densely
  DevBuf<double> dense, dense_rows, dense_gather, crhs, cgather, cglob, csol;
  DevBuf<int32_t> coff, ccolmap;
  int32_t cN = 0, cnmax = 0, coff_me = 0;
  DevBuf<int> info;
  bool dense_coarse = false;
  bool built = false;
  double op_complexity = 0.0;
  Reducer red;
  // Chebyshev smoother: per level the bound of lambda_max(D^-1 A) being reduced, the value in use and the
  // coefficients made from it (amg_cheby_coef_kernel; coef_stride doubles per level)
  DevBuf<double> lmax_bound, lmax, coef;
  int coef_stride = 0, coef_sweeps = 0;
  DevBuf<double> fixed_coef;   // {c1, c2} of launch_level_smoother
  // the V-cycle as a CUDA graph: one launch instead of ~100 kernel launches + ~35 NCCL calls
  cudaGraphExec_t gexec = nullptr;
  bool graph_valid = false;    // false after a refresh of the hierarchy
  const void* graph_key[5] = {};   // buffers of the fine matrix the captured graph reads
  bool graph_seams = false;        // the captured cycle leaves its first and last fine step to Amg::apply
  const float* exit_x = nullptr;   // seams: the iterate the last fine sweep (amg_cheby_kernel<CHEBY_EXIT>) reads
  bool warm = false;           // one plain cycle after a (re)build so that lazy allocations are done
  int64_t graph_launches = 0;  // kernels inside the graph (for the launch accounting)
  void* result_ptr = nullptr;  // where level 0's solution ends up
  // ---- replicated coarse part (multi-GPU).  Below ~1e5 rows a level is pure latency: a handful of
  // microsecond kernels separated by halo exchanges.  From `tail_level` on, every rank therefore holds
  // the WHOLE level (values all-gathered at each refresh) and a complete serial sub-hierarchy `tail`
  // built from it -- identical on all ranks, no communication.  Per V-cycle one all-gather of the
  // level's right-hand side remains; the prolongation above it needs no exchange because every rank has
  // the whole coarse solution.
  int tail_level = -1;
  std::unique_ptr<Amg> tail;
  HostCsr tailA;                 // global pattern of the level (rows and columns in global numbering)
  HostSell tailS;
  DevSell tailM;                 // its values
  DevBuf<int32_t> tail_diag;     // SELL positions of the diagonal
  int32_t tail_N = 0, tail_nmax = 0, tail_wmax = 0;
  DevBuf<int32_t> tail_pack_pos;     // [n][wmax] of my rows: position in the level's SELL values (or -1)
  DevBuf<int32_t> tail_unpack_pos;   // [rank][nmax][wmax]: position in tailM.val (or -1)
  DevBuf<double> tail_send, tail_recv;
  DevBuf<int32_t> tail_gid;          // local column (own + ghost) of the level -> global row id
  DevBuf<int32_t> tail_off;          // first global id of every rank (n_ranks + 1)
  HaloPlan tail_halo;                // empty plan handed to the (serial) tail
  std::vector<Neighbor> no_nbrs;
  int sm_count = 148;
  P2pGather tail_gather;             // right-hand side all-gather through the symmetric heap
  DevBuf<double> tail_rhs_d, tail_gather_d;   // NCCL fallback: padded blocks
  ~Impl() {
    if (gexec) cudaGraphExecDestroy(gexec);
  }
};

Amg::Amg() : p_(new Impl()) {}
Amg::~Amg() = default;
int Amg::levels() const { return (int)p_->lv.size() + (p_->tail ? p_->tail->levels() - 1 : 0); }
bool Amg::fp32() const { return p_->opt.fp32_cycle != 0; }
double Amg::operator_complexity() const { return p_->op_complexity; }

static std::vector<int32_t> diag_positions(const HostCsr& A, const HostSell& S, int32_t n) {
  std::vector<int32_t> d(n, 0);
  for (int32_t r = 0; r < n; ++r) {
    const int32_t* b = A.col.data() + A.rowptr[r];
    const int32_t* e = A.col.data() + A.rowptr[r + 1];
    const int32_t* p = std::lower_bound(b, e, r);
    if (p == e || *p != r) throw Error(SHAKTI_ERR_INVALID, "AMG: matrix row without diagonal entry");
    d[r] = (int32_t)S.pos(r, (int)(p - b));
  }
  return d;
}

void Amg::setup(const HostCsr& A0, const HostSell& S0, const std::vector<uint8_t>& exclude, const std::vector<Neighbor>& nbrs,
                HaloPlan* halo, const AmgOptions& opt, int sm_count, cudaStream_t s) {
  Impl& I = *p_;
  I.opt = opt;
  I.s = s;
  I.A0 = &A0;
  I.S0 = &S0;
  I.nbrs0 = &nbrs;
  I.halo0 = halo;
  I.exclude = exclude;
  I.lv.clear();
  I.built = false;
  I.graph_valid = false;
  I.warm = false;
  I.red.init(sm_count);
  I.sm_count = sm_count;
  I.tail.reset();
  I.tail_level = -1;
  I.fixed_coef.upload(std::vector<double>{0.3, 0.2});
  refreshes_ = 0;
}

template <class T>
static void alloc_cycle_vectors(CycleVecs<T>& v, const AmgLevel& L, cudaStream_t s) {
  v.x.alloc_zero(std::max(L.n_cols, 1), s);
  v.x2.alloc_zero(std::max(L.n_cols, 1), s);
  v.b.alloc_zero(std::max(L.n, 1), s);
  v.r.alloc_zero(std::max(L.n, 1), s);
  v.d.alloc_zero(std::max(L.n, 1), s);
  v.dinv.alloc_zero(std::max(L.n, 1), s);
}
static void alloc_level_vectors(AmgLevel& L, bool fp32, cudaStream_t s) {
  L.dinv.alloc_zero(std::max(L.n, 1), s);
  if (fp32) alloc_cycle_vectors(L.vf, L, s);
  else alloc_cycle_vectors(L.vd, L, s);
}
template <class T> static CycleVecs<T>& vecs(AmgLevel& L);
template <> CycleVecs<double>& vecs<double>(AmgLevel& L) { return L.vd; }
template <> CycleVecs<float>& vecs<float>(AmgLevel& L) { return L.vf; }

// numeric phase of one level: smoother diagonal, P (own rows, then the neighbours' interface
// rows by halo exchange), R, AP and the next level's operator
static void numeric_level(Amg::Impl& I, size_t l, const DevSell& Afine, const int32_t* fine_diag_pos) {
  cudaStream_t s = I.s;
  AmgLevel& L = *I.lv[l];
  const DevSell& A = (l == 0) ? Afine : L.A;
  const int32_t* dpos = (l == 0) ? fine_diag_pos : L.diag_pos.p;
  if (L.n > 0) SHAKTI_LAUNCH(amg_dinv_kernel, div_up(L.n, 256), 256, 0, s, L.n, dpos, A.val.p, L.dinv.p);
  if (L.last) return;
  SHAKTI_CUDA(cudaMemsetAsync(L.P.val.p, 0, sizeof(double) * L.P.padded, s));
  if (L.n > 0)
    SHAKTI_LAUNCH(amg_prolongator_kernel, div_up(L.n, 256), 256, 0, s, view(A), L.pmap.p, dpos, L.dinv.p,
                  I.opt.prolong_omega, L.P.slice_ptr.p, L.P.val.p);
  if (comm().active() && L.maxw > 0) {
    const int64_t ns = (int64_t)L.halo->n_send_total() * L.maxw, ng = (int64_t)L.n_ghost * L.maxw;
    if (ns) SHAKTI_LAUNCH(amg_pack_rows_kernel, div_up(ns, 256), 256, 0, s, ns, L.psend_pos.p, L.P.val.p, L.psend.p);
    L.halo->exchange_packed(L.psend.p, L.precv.p, L.n, L.maxw, s);
    if (ng) SHAKTI_LAUNCH(amg_unpack_rows_kernel, div_up(ng, 256), 256, 0, s, ng, L.pg_pos.p, L.precv.p, L.P.val.p);
  }
  if (L.R.padded)
    SHAKTI_LAUNCH(amg_gather_vals_kernel, (int)std::min<int64_t>(148 * 8, std::max<int64_t>(1, (L.R.padded + 255) / 256)), 256, 0, s,
                  L.R.padded, L.tmap.p, L.P.val.p, L.R.val.p);
  spgemm_numeric(A, L.P, L.AP, L.plan_AP, s);                 // A restricted to the columns P has rows for
  spgemm_numeric(L.R, L.AP, I.lv[l + 1]->A, L.plan_RAP, s);    // Galerkin: R (A P)
}

static bool uses_half(const Amg::Impl& I, const DevSell& A) {
  // Opt-in (SHAKTI_AMG_FP16=1).  Measured at C4: the fine-level smoother goes from 270 to 257 us (-5 %) for 17 % fewer
  // bytes -- at 6 B per entry the kernel is no longer purely HBM bound (0.66 instead of 0.76 of the measured peak; the
  // x gathers set the pace) -- and a time step from 96.5 to 94.6 ms with unchanged iteration counts.
  static const bool on = getenv("SHAKTI_AMG_FP16") != nullptr && atoi(getenv("SHAKTI_AMG_FP16")) != 0;
  return on && I.opt.fp32_cycle && I.opt.smoother == 1 && A.n_rows >= kChebyWideRowsBelow;
}

// Copies the V-cycle reads: smoother diagonal in the cycle's precision and, for the mixed-precision
// cycle, single-precision values of A, P and R (half-precision row-scaled values of A on the large levels).
// fine_done: level 0's diagonal and A were copied by fine_refresh_pass.
static void sync_cycle_precision(Amg::Impl& I, size_t l, const DevSell& Afine, bool matrices, bool fine_done = false) {
  cudaStream_t s = I.s;
  AmgLevel& L = *I.lv[l];
  const DevSell& A = (l == 0) ? Afine : L.A;
  if (I.opt.fp32_cycle) {
    if (!(l == 0 && fine_done)) {
      launch_d2f(L.n, L.dinv.p, L.vf.dinv.p, s);
      if (uses_half(I, A)) A.refresh_f16_scaled(L.dinv.p, s);
      else A.refresh_f32(s);
    }
    if (matrices && !L.last) { L.P.refresh_f32(s); L.R.refresh_f32(s); }
  } else if (L.n) {
    SHAKTI_CUDA(cudaMemcpyAsync(L.vd.dinv.p, L.dinv.p, sizeof(double) * L.n, cudaMemcpyDeviceToDevice, s));
  }
}

// Level 0 takes the one-pass refresh (amg_fine_refresh_kernel) when it needs both what that pass fuses: the
// copies of the mixed-precision cycle and the Chebyshev bound.
static bool fine_one_pass(const Amg::Impl& I) { return I.opt.fp32_cycle && I.opt.smoother == 1 && I.lv[0]->n > 0; }

// dinv (fp64, fp32), the cycle's copy of the fine values and level 0's bound (atomic maximum into `bound`, zeroed
// by the caller) in one pass; the half-precision copy, where level 0 uses one, is made from dinv afterwards
static void fine_refresh_pass(Amg::Impl& I, const DevSell& Afine, const int32_t* fine_diag_pos, double* bound) {
  cudaStream_t s = I.s;
  AmgLevel& L = *I.lv[0];
  unsigned long long* b = reinterpret_cast<unsigned long long*>(bound);
  const int grid = bound_blocks((int64_t)Afine.n_slices * 32, I.sm_count);
  if (uses_half(I, Afine)) {
    SHAKTI_LAUNCH(amg_fine_refresh_kernel<false>, grid, 256, 0, s, view(Afine), fine_diag_pos, L.dinv.p, L.vf.dinv.p, nullptr, b);
    Afine.refresh_f16_scaled(L.dinv.p, s);
  } else {
    if (Afine.valf.n != (size_t)Afine.padded) Afine.valf.alloc((size_t)Afine.padded);
    SHAKTI_LAUNCH(amg_fine_refresh_kernel<true>, grid, 256, 0, s, view(Afine), fine_diag_pos, L.dinv.p, L.vf.dinv.p, Afine.valf.p, b);
  }
}

static void launch_cheby_coef(Amg::Impl& I, int nl, bool keep) {
  SHAKTI_LAUNCH(amg_cheby_coef_kernel, 1, 32, 0, I.s, nl, I.coef_sweeps, I.coef_stride, I.opt.cheby_ratio, I.lmax_bound.p,
                keep ? 1 : 0, I.lmax.p, I.coef.p);
}

// Upper end of the spectrum of D^-1 A for the Chebyshev smoother, recomputed at every refresh: the
// Gershgorin number max_i sum_j |a_ij| / |a_ii| -- one pass per level, identical on every rank, turned
// into the smoother's coefficients on the device.  It is a guaranteed upper bound.  (Round-1 history: 1.1 x
// a warm-started power-iteration estimate is ~4 % faster at 16M dofs but under-estimates after large changes
// of the operator, which makes the smoother amplify the top of the spectrum and stalled the Krylov solve on
// a small case; a bound cannot do that.)  Returns whether level 0 went through fine_refresh_pass.
static bool update_smoother_bounds(Amg::Impl& I, const DevSell& Afine, const int32_t* fine_diag_pos) {
  cudaStream_t s = I.s;
  const size_t nl = I.lv.size();
  if (I.opt.smoother != 1) return false;
  if (I.lmax_bound.n < nl) {
    // sized once per hierarchy, before the first capture of the V-cycle
    I.coef_sweeps = std::max({I.opt.presmooth, I.opt.postsmooth, 8});
    I.coef_stride = 2 + 2 * I.coef_sweeps;
    I.lmax_bound.alloc_zero(nl, s);
    I.lmax.alloc_zero(nl, s);
    I.coef.alloc_zero(nl * I.coef_stride, s);
  }
  SHAKTI_CUDA(cudaMemsetAsync(I.lmax_bound.p, 0, sizeof(double) * nl, s));
  const bool fine = fine_one_pass(I);
  for (size_t l = 0; l < nl; ++l) {
    AmgLevel& L = *I.lv[l];
    if (l == 0 && fine) fine_refresh_pass(I, Afine, fine_diag_pos, I.lmax_bound.p);
    else if (L.n > 0)
      SHAKTI_LAUNCH(amg_gershgorin_kernel, bound_blocks(L.n, I.sm_count), 256, 0, s, view(l == 0 ? Afine : L.A), L.dinv.p,
                    reinterpret_cast<unsigned long long*>(I.lmax_bound.p + l));
  }
  comm_allreduce_max(I.lmax_bound.p, (int)nl, s);
  launch_cheby_coef(I, (int)nl, false);
  return fine;
}

// One coarsening step on the host: rank-local aggregation on strong connections, prolongator
// pattern over own + ghost aggregates, the neighbours' interface rows of P, R = (P[own,own])^T,
// the two product patterns and the halo plan of the coarse level.
static void coarsen_level(Amg::Impl& I, size_t l, const DevSell& dA, const HostCsr& A, const HostSell& S,
                          const std::vector<uint8_t>& excl, bool& stalled) {
  cudaStream_t s = I.s;
  const AmgOptions& opt = I.opt;
  AmgLevel& L = *I.lv[l];
  const int me = comm().rank, nranks = comm().nranks;
  const int32_t n = L.n, g = L.n_ghost;
  // ---- strength + aggregation (own rows, own columns)
  std::vector<uint8_t> strong;
  const double theta = opt.strength_theta * std::pow(0.5, (double)l);
  if (theta > 0 && n > 0) {
    std::vector<double> v = dA.val.download(s);
    std::vector<double> diag(n, 0.0);
    for (int32_t i = 0; i < n; ++i)
      for (int32_t k = A.rowptr[i]; k < A.rowptr[i + 1]; ++k)
        if (A.col[k] == i) diag[i] = std::fabs(v[S.pos(i, k - A.rowptr[i])]);
    strong.assign(A.nnz(), 0);
    for (int32_t i = 0; i < n; ++i)
      for (int32_t k = A.rowptr[i]; k < A.rowptr[i + 1]; ++k) {
        const int32_t j = A.col[k];
        if (j >= n || j == i) continue;
        const double a = std::fabs(v[S.pos(i, k - A.rowptr[i])]);
        strong[k] = (a >= theta * std::sqrt(diag[i] * diag[j])) && a > 0;
      }
  }
  std::vector<int32_t> agg;
  const int32_t nc = n > 0 ? aggregate(A, n, excl, strong, agg) : 0;
  const double nc_glob = comm_host_sum((double)nc, s), n_glob = comm_host_sum((double)n, s);
  if (nc_glob <= 0 || nc_glob > 0.85 * n_glob) { stalled = true; return; }
  stalled = false;
  L.n_coarse = nc;
  // ---- aggregate of every ghost column: (owner rank, index on the owner) or none
  std::vector<int> gowner(g, -1);
  for (const auto& nb : L.nbrs)
    for (int32_t k = 0; k < nb.recv_count; ++k) gowner[nb.recv_begin - n + k] = nb.rank;
  std::vector<double> gagg(g, -1.0);
  if (comm().active()) {
    std::vector<double> tmp((size_t)n + g, -1.0);
    for (int32_t i = 0; i < n; ++i) tmp[i] = (double)agg[i];
    DevBuf<double> dv;
    dv.upload(tmp);
    L.halo->exchange(dv.p, s);
    tmp = dv.download(s);
    for (int32_t k = 0; k < g; ++k) gagg[k] = tmp[n + k];
  }
  typedef std::pair<int, int32_t> Gid;          // (rank, index on that rank)
  auto gid_of_col = [&](int32_t j) -> Gid {      // aggregate of local column j, (-1,-1) if none
    if (j < n) return agg[j] >= 0 ? Gid(me, agg[j]) : Gid(-1, -1);
    const double a = gagg[j - n];
    return a >= 0 ? Gid(gowner[j - n], (int32_t)a) : Gid(-1, -1);
  };
  // ---- prolongator rows of own vertices in global aggregate ids
  const bool smoothed = opt.prolong_omega != 0.0;
  std::vector<std::vector<Gid>> prow((size_t)n + g);
  for (int32_t i = 0; i < n; ++i) {
    if (agg[i] < 0) continue;
    auto& r = prow[i];
    if (smoothed) {
      for (int32_t k = A.rowptr[i]; k < A.rowptr[i + 1]; ++k) {
        const Gid c = gid_of_col(A.col[k]);
        if (c.first >= 0) r.push_back(c);
      }
      std::sort(r.begin(), r.end());
      r.erase(std::unique(r.begin(), r.end()), r.end());
    } else {
      r.push_back(Gid(me, agg[i]));
    }
  }
  // ---- interface rows of the neighbours (pattern exchange, fixed width)
  int maxw = 0;
  const std::vector<int32_t>& sidx = L.halo->send_idx_host;
  for (int32_t v : sidx) maxw = std::max<int>(maxw, (int)prow[v].size());
  maxw = (int)comm_host_max((double)maxw, s);
  L.maxw = comm().active() ? maxw : 0;
  if (comm().active() && maxw > 0) {
    const int wp = 1 + 2 * maxw;
    std::vector<double> sb((size_t)std::max<size_t>(sidx.size(), 1) * wp, -1.0), rb((size_t)std::max(g, 1) * wp, -1.0);
    for (size_t k = 0; k < sidx.size(); ++k) {
      const auto& r = prow[sidx[k]];
      sb[k * wp] = (double)r.size();
      for (size_t w = 0; w < r.size(); ++w) { sb[k * wp + 1 + 2 * w] = r[w].first; sb[k * wp + 2 + 2 * w] = r[w].second; }
    }
    DevBuf<double> dsb, drb;
    dsb.upload(sb);
    drb.upload(rb);
    L.halo->exchange_packed(dsb.p, drb.p, n, wp, s);
    rb = drb.download(s);
    for (int32_t k = 0; k < g; ++k) {
      const int len = (int)rb[(size_t)k * wp];
      for (int w = 0; w < len; ++w)
        prow[(size_t)n + k].push_back(Gid((int)rb[(size_t)k * wp + 1 + 2 * w], (int32_t)rb[(size_t)k * wp + 2 + 2 * w]));
      // NOTE: kept in the owner's order; slot w of the value exchange refers to this order
    }
  }
  // ---- ghost aggregates: everything referenced that is not mine, sorted by (owner, index)
  std::vector<Gid> gset;
  for (const auto& r : prow)
    for (const Gid& c : r)
      if (c.first != me) gset.push_back(c);
  std::sort(gset.begin(), gset.end());
  gset.erase(std::unique(gset.begin(), gset.end()), gset.end());
  const int32_t gc = (int32_t)gset.size();
  L.n_coarse_ghost = gc;
  auto local_col = [&](const Gid& c) -> int32_t {
    if (c.first == me) return c.second;
    return nc + (int32_t)(std::lower_bound(gset.begin(), gset.end(), c) - gset.begin());
  };
  // ---- P (n + g rows) with sorted local columns; remember where the exchanged values go
  HostCsr P;
  P.n_rows = (int64_t)n + g;
  P.n_cols = (int64_t)nc + gc;
  P.rowptr.assign(P.n_rows + 1, 0);
  std::vector<std::vector<int32_t>> order((size_t)g);   // ghost rows: slot w -> rank in sorted row
  {
    std::vector<std::pair<int32_t, int>> tmp;
    for (int64_t i = 0; i < P.n_rows; ++i) {
      tmp.clear();
      for (size_t w = 0; w < prow[i].size(); ++w) tmp.push_back({local_col(prow[i][w]), (int)w});
      std::sort(tmp.begin(), tmp.end());
      if (i >= n) order[i - n].assign(tmp.size(), 0);
      for (size_t q = 0; q < tmp.size(); ++q) {
        P.col.push_back(tmp[q].first);
        if (i >= n) order[i - n][tmp[q].second] = (int32_t)q;
      }
      P.rowptr[i + 1] = (int32_t)P.col.size();
    }
  }
  HostSell PS = sell_from_csr(P);
  // pmap: A entry (i,j) -> position of aggregate(j) inside P's row i
  {
    std::vector<uint8_t> pm(S.padded(), 255);
    for (int32_t i = 0; i < n; ++i) {
      const int32_t* pb = P.col.data() + P.rowptr[i];
      const int32_t* pe = P.col.data() + P.rowptr[i + 1];
      if (pb == pe) continue;
      for (int32_t k = A.rowptr[i]; k < A.rowptr[i + 1]; ++k) {
        const int32_t j = A.col[k];
        if (!smoothed && j != i) continue;
        const Gid c = gid_of_col(j);
        if (c.first < 0) continue;
        const int32_t* q = std::lower_bound(pb, pe, local_col(c));
        const int64_t t = q - pb;
        if (t > 254) throw Error(SHAKTI_ERR_INVALID, "AMG: prolongator row too long");
        pm[S.pos(i, k - A.rowptr[i])] = (uint8_t)t;
      }
    }
    L.pmap.upload(pm);
  }
  L.P.upload_pattern(PS, P.nnz());
  if (L.maxw > 0) {
    // own interface rows: slot w of send entry k = w-th entry of the (sorted-by-Gid) own row; own rows were
    // built sorted by Gid, and local_col is monotone in Gid only per owner, so map through the sorted order
    std::vector<int32_t> sp((size_t)std::max<size_t>(sidx.size(), 1) * L.maxw, -1), gp((size_t)std::max(g, 1) * L.maxw, -1);
    for (size_t k = 0; k < sidx.size(); ++k) {
      const int32_t i = sidx[k];
      const int32_t* pb = P.col.data() + P.rowptr[i];
      const int32_t* pe = P.col.data() + P.rowptr[i + 1];
      for (size_t w = 0; w < prow[i].size(); ++w) {
        const int32_t* q = std::lower_bound(pb, pe, local_col(prow[i][w]));
        sp[k * L.maxw + w] = (int32_t)PS.pos(i, (int)(q - pb));
      }
    }
    for (int32_t k = 0; k < g; ++k)
      for (size_t w = 0; w < order[k].size(); ++w) gp[(size_t)k * L.maxw + w] = (int32_t)PS.pos((int64_t)n + k, order[k][w]);
    L.psend_pos.upload(sp);
    L.pg_pos.upload(gp);
    L.psend.alloc_zero(sp.size(), s);
    L.precv.alloc_zero(gp.size(), s);
  }
  // ---- R = transpose of the own-rows x own-aggregates block of P
  HostCsr Pown;
  Pown.n_rows = n;
  Pown.n_cols = nc;
  Pown.rowptr.assign((size_t)n + 1, 0);
  std::vector<int32_t> pown_entry;   // entry of P for each entry of Pown
  for (int32_t i = 0; i < n; ++i) {
    for (int32_t k = P.rowptr[i]; k < P.rowptr[i + 1]; ++k)
      if (P.col[k] < nc) { Pown.col.push_back(P.col[k]); pown_entry.push_back(k); }
    Pown.rowptr[i + 1] = (int32_t)Pown.col.size();
  }
  std::vector<int32_t> tentry;
  HostCsr R = csr_transpose(Pown, &tentry);
  HostSell RS = sell_from_csr(R);
  {
    std::vector<int32_t> ppos = sell_positions(P, PS);
    std::vector<int32_t> tm(RS.padded(), -1);
    for (int64_t r = 0; r < R.n_rows; ++r)
      for (int32_t k = R.rowptr[r]; k < R.rowptr[r + 1]; ++k) tm[RS.pos(r, k - R.rowptr[r])] = ppos[pown_entry[tentry[k]]];
    L.tmap.upload(tm);
  }
  L.R.upload_pattern(RS, R.nnz());
  // ---- product patterns
  HostCsr AP = product_pattern(A, P);
  L.AP.upload_pattern(sell_from_csr(AP), AP.nnz());
  std::unique_ptr<AmgLevel> Ln(new AmgLevel());
  Ln->hA = product_pattern(R, AP);
  Ln->hA.n_cols = (int64_t)nc + gc;
  Ln->hS = sell_from_csr(Ln->hA);
  Ln->index = (int32_t)l + 1;
  Ln->n = nc;
  Ln->n_ghost = gc;
  Ln->n_cols = nc + gc;
  Ln->nnz = Ln->hA.nnz();
  Ln->A.upload_pattern(Ln->hS, Ln->hA.nnz());
  Ln->diag_pos.upload(diag_positions(Ln->hA, Ln->hS, nc));
  // ---- halo plan of the coarse level: ask every owner for the aggregates referenced here
  if (comm().active()) {
    std::vector<std::vector<double>> ask(nranks);
    std::vector<int32_t> rb(nranks, 0), rc(nranks, 0);
    for (int32_t k = 0; k < gc; ++k) {
      const int o = gset[k].first;
      if (rc[o] == 0) rb[o] = nc + k;
      rc[o]++;
      ask[o].push_back((double)gset[k].second);
    }
    std::vector<std::vector<double>> asked = comm_exchange_lists(ask, s);
    for (int r = 0; r < nranks; ++r) {
      if (r == me || (asked[r].empty() && rc[r] == 0)) continue;
      Neighbor nb;
      nb.rank = r;
      for (double v : asked[r]) nb.send_local.push_back((int32_t)v);
      nb.recv_begin = rb[r];
      nb.recv_count = rc[r];
      Ln->nbrs.push_back(std::move(nb));
    }
  }
  Ln->own_halo.build(Ln->nbrs);
  Ln->halo = &Ln->own_halo;
  alloc_level_vectors(*Ln, I.opt.fp32_cycle != 0, s);
  I.lv.push_back(std::move(Ln));
}

// Makes level l the root of the replicated part of the hierarchy (see Amg::Impl::tail): gathers the
// level's pattern from all ranks in a global numbering (ranks in order), builds the maps that move its
// values at every refresh, and sets up a serial Amg on it.
static void build_tail(Amg::Impl& I, size_t l) {
  cudaStream_t s = I.s;
  AmgLevel& L = *I.lv[l];
  const HostCsr& A = (l == 0) ? *I.A0 : L.hA;
  const HostSell& S = (l == 0) ? *I.S0 : L.hS;
  const int me = comm().rank, nr = comm().nranks;
  const int32_t n = L.n;
  const std::vector<double> counts = comm_host_allgather((double)n, s);
  std::vector<int32_t> off(nr + 1, 0), cnt(nr, 0);
  int32_t nmax = 1;
  for (int r = 0; r < nr; ++r) {
    cnt[r] = (int32_t)counts[r];
    off[r + 1] = off[r] + cnt[r];
    nmax = std::max(nmax, cnt[r]);
  }
  const int32_t N = off[nr];
  // global id of every local column: own rows by offset, ghosts from their owners
  std::vector<int32_t> gid(std::max(L.n_cols, 1), 0);
  {
    std::vector<double> tmp((size_t)std::max(L.n_cols, 1), 0.0);
    for (int32_t c = 0; c < n; ++c) tmp[c] = (double)(off[me] + c);
    DevBuf<double> dv;
    dv.upload(tmp);
    L.halo->exchange(dv.p, s);
    tmp = dv.download(s);
    for (int32_t c = 0; c < L.n_cols; ++c) gid[c] = (int32_t)tmp[c];
  }
  int32_t wloc = 1;
  for (int32_t i = 0; i < n; ++i) wloc = std::max(wloc, A.rowptr[i + 1] - A.rowptr[i]);
  const int32_t wmax = (int32_t)comm_host_max((double)wloc, s);
  // my rows (length, then global columns in local CSR order) to every rank
  std::vector<double> mine;
  mine.reserve((size_t)n + A.nnz());
  for (int32_t i = 0; i < n; ++i) {
    mine.push_back((double)(A.rowptr[i + 1] - A.rowptr[i]));
    for (int32_t k = A.rowptr[i]; k < A.rowptr[i + 1]; ++k) mine.push_back((double)gid[A.col[k]]);
  }
  const std::vector<std::vector<double>> in = comm_exchange_lists(std::vector<std::vector<double>>(nr, mine), s);
  HostCsr& G = I.tailA;
  G = HostCsr();
  G.n_rows = G.n_cols = N;
  G.rowptr.assign((size_t)N + 1, 0);
  std::vector<int32_t> order;   // for every gathered entry (rank-major, CSR order): its place in the sorted global row
  std::vector<std::pair<int32_t, int32_t>> tmp;
  for (int r = 0; r < nr; ++r) {
    const std::vector<double>& v = in[r];
    size_t p = 0;
    for (int32_t i = 0; i < cnt[r]; ++i) {
      const int len = (int)v[p++];
      tmp.clear();
      for (int k = 0; k < len; ++k) tmp.push_back({(int32_t)v[p++], k});
      std::sort(tmp.begin(), tmp.end());
      const size_t base = order.size();
      order.resize(base + len);
      for (int q = 0; q < len; ++q) {
        G.col.push_back(tmp[q].first);
        order[base + tmp[q].second] = q;
      }
      G.rowptr[(size_t)off[r] + i + 1] = (int32_t)G.col.size();
    }
  }
  I.tailS = sell_from_csr(G);
  std::vector<int32_t> unpack((size_t)nr * nmax * wmax, -1), pack((size_t)nmax * wmax, -1);
  {
    size_t e = 0;
    for (int r = 0; r < nr; ++r)
      for (int32_t i = 0; i < cnt[r]; ++i) {
        const int32_t gr = off[r] + i;
        const int len = G.rowptr[gr + 1] - G.rowptr[gr];
        for (int k = 0; k < len; ++k, ++e) unpack[((size_t)r * nmax + i) * wmax + k] = (int32_t)I.tailS.pos(gr, order[e]);
      }
  }
  for (int32_t i = 0; i < n; ++i)
    for (int32_t k = A.rowptr[i]; k < A.rowptr[i + 1]; ++k) pack[(size_t)i * wmax + (k - A.rowptr[i])] = (int32_t)S.pos(i, k - A.rowptr[i]);
  I.tail_N = N; I.tail_nmax = nmax; I.tail_wmax = wmax;
  I.tail_pack_pos.upload(pack);
  I.tail_unpack_pos.upload(unpack);
  I.tail_send.alloc_zero((size_t)nmax * wmax, s);
  I.tail_recv.alloc_zero((size_t)nr * nmax * wmax, s);
  I.tail_gid.upload(gid);
  I.tail_off.upload(off);
  I.tailM.upload_pattern(I.tailS, G.nnz());
  I.tail_diag.upload(diag_positions(G, I.tailS, N));
  if (comm().p2p) {
    I.tail_gather.build(nmax, s);
    I.tail_gather.set_counts(cnt);
  } else {
    I.tail_rhs_d.alloc_zero(nmax, s);
    I.tail_gather_d.alloc_zero((size_t)nr * nmax, s);
  }
  AmgOptions to = I.opt;
  to.cuda_graph = 0;   // its kernels are captured as part of the distributed cycle's graph
  I.tail.reset(new Amg());
  I.tail_level = (int)l;
  {
    CommSerialScope serial;
    I.tail->setup(I.tailA, I.tailS, std::vector<uint8_t>(), I.no_nbrs, &I.tail_halo, to, I.sm_count, s);
  }
}

// all-gather the replicated level's values and renew the serial sub-hierarchy below it
static void refresh_tail(Amg::Impl& I, const DevSell& Afine) {
  if (!I.tail) return;
  cudaStream_t s = I.s;
  const DevSell& A = (I.tail_level == 0) ? Afine : I.lv[I.tail_level]->A;
  const int64_t blk = (int64_t)I.tail_nmax * I.tail_wmax;
  SHAKTI_LAUNCH(amg_pack_rows_kernel, div_up(blk, 256), 256, 0, s, blk, I.tail_pack_pos.p, A.val.p, I.tail_send.p);
  comm_allgather(I.tail_send.p, I.tail_recv.p, (int)blk, s);
  const int64_t tot = blk * comm().nranks;
  SHAKTI_LAUNCH(amg_unpack_rows_kernel, div_up(tot, 256), 256, 0, s, tot, I.tail_unpack_pos.p, I.tail_recv.p, I.tailM.val.p);
  CommSerialScope serial;
  I.tail->refresh(I.tailM, I.tail_diag.p);
}

static void build_hierarchy(Amg::Impl& I, const DevSell& Afine, const int32_t* fine_diag_pos) {
  cudaStream_t s = I.s;
  const AmgOptions& opt = I.opt;
  I.lv.clear();
  {
    std::unique_ptr<AmgLevel> L0(new AmgLevel());
    L0->n = (int32_t)I.A0->n_rows;
    L0->n_cols = (int32_t)I.A0->n_cols;
    L0->n_ghost = L0->n_cols - L0->n;
    L0->nnz = I.A0->nnz();
    L0->nbrs = *I.nbrs0;
    L0->halo = I.halo0;
    alloc_level_vectors(*L0, I.opt.fp32_cycle != 0, s);
    I.lv.push_back(std::move(L0));
  }
  std::vector<uint8_t> excl = I.exclude;
  double nnz_sum = 0.0;
  for (size_t l = 0;; ++l) {
    AmgLevel& L = *I.lv[l];
    const HostCsr& A = (l == 0) ? *I.A0 : L.hA;
    const HostSell& S = (l == 0) ? *I.S0 : L.hS;
    const DevSell& dA = (l == 0) ? Afine : L.A;
    nnz_sum += (double)A.nnz();
    const double n_glob = comm_host_sum((double)L.n, s);
    bool stop = (n_glob <= opt.coarse_size) || ((int)l + 1 >= opt.max_levels);
    // multi-GPU: small levels are replicated (at the latest the level where coarsening ends, unless it is huge)
    if (comm().active() && n_glob <= std::max(opt.replicate_below, opt.coarse_size)) {
      build_tail(I, l);
      L.last = true;
      numeric_level(I, l, Afine, fine_diag_pos);
      break;
    }
    bool stalled = false;
    if (!stop) coarsen_level(I, l, dA, A, S, excl, stalled);
    if (stop || stalled) {
      if (comm().active() && n_glob <= 4.0e6) build_tail(I, l);
      L.last = true;
      numeric_level(I, l, Afine, fine_diag_pos);
      break;
    }
    numeric_level(I, l, Afine, fine_diag_pos);
    excl.clear();
  }
  // ---- coarsest level: gather on every rank, invert densely
  AmgLevel& last = *I.lv.back();
  const std::vector<double> counts = comm_host_allgather((double)last.n, s);
  int64_t N = 0, nmax = 0;
  std::vector<int32_t> off(counts.size() + 1, 0);
  for (size_t r = 0; r < counts.size(); ++r) {
    off[r + 1] = off[r] + (int32_t)counts[r];
    nmax = std::max<int64_t>(nmax, (int64_t)counts[r]);
  }
  N = off.back();
  I.dense_coarse = N <= 1024 && N > 0 && !I.tail;
  if (I.dense_coarse) {
    const int me = comm().rank, nr = comm().nranks;
    I.cN = (int32_t)N;
    I.cnmax = (int32_t)nmax;
    I.coff_me = off[me];
    I.coff.upload(off);
    std::vector<int32_t> colmap(std::max(last.n_cols, 1), 0);
    for (int32_t c = 0; c < last.n; ++c) colmap[c] = off[me] + c;
    if (last.n_ghost > 0) {
      // ghost column -> (owner, index on owner): recorded when the level was created (its nbrs lists give the owner,
      // the index is recovered by asking the owners, exactly as for the halo plan)
      std::vector<double> tmp((size_t)last.n_cols, 0.0);
      for (int32_t c = 0; c < last.n; ++c) tmp[c] = (double)(off[me] + c);
      DevBuf<double> dv;
      dv.upload(tmp);
      last.halo->exchange(dv.p, s);
      tmp = dv.download(s);
      for (int32_t c = last.n; c < last.n_cols; ++c) colmap[c] = (int32_t)tmp[c];
    }
    I.ccolmap.upload(colmap);
    I.dense.alloc_zero((size_t)2 * N * N, s);
    I.dense_rows.alloc_zero((size_t)std::max<int64_t>(nmax, 1) * N, s);
    I.dense_gather.alloc_zero((size_t)nr * std::max<int64_t>(nmax, 1) * N, s);
    I.crhs.alloc_zero(std::max<int64_t>(nmax, 1), s);
    I.cgather.alloc_zero((size_t)nr * std::max<int64_t>(nmax, 1), s);
    I.cglob.alloc_zero(N, s);
    I.csol.alloc_zero(N, s);
    I.info.alloc_zero(1, s);
  }
  const double nnz0 = comm_host_sum((double)I.A0->nnz(), s);
  nnz_sum = comm_host_sum(nnz_sum, s);
  I.op_complexity = nnz0 > 0 ? nnz_sum / nnz0 : 0.0;
  I.built = true;
  if (I.tail) {
    // the tail's own hierarchy is built by its first refresh (values needed): done right away so that the
    // level count and the complexity are final when this returns
    refresh_tail(I, Afine);
    const double nnz_root = (double)I.tailA.nnz();
    if (nnz0 > 0) I.op_complexity += (I.tail->operator_complexity() - 1.0) * nnz_root / nnz0;
  }
}

// Cheap per-solve update when the hierarchy itself is kept (lagged): the fine-level smoother must
// match the CURRENT operator, so its diagonal is recomputed and its Chebyshev bound is set to the
// (always safe) Gershgorin bound.  Coarse levels stay consistent among themselves.  Everything stays on
// the device and no kernel argument changes, so the captured V-cycle is replayed as it is.
void Amg::refresh_fine_smoother(const DevSell& Afine, const int32_t* fine_diag_pos) {
  Impl& I = *p_;
  cudaStream_t s = I.s;
  if (!I.built || I.lv.empty()) return;
  AmgLevel& L = *I.lv[0];
  const bool cheby = I.opt.smoother == 1 && !(L.last && I.dense_coarse);
  if (cheby) SHAKTI_CUDA(cudaMemsetAsync(I.lmax_bound.p, 0, sizeof(double), s));
  const bool fine = cheby && fine_one_pass(I);
  if (fine) {
    fine_refresh_pass(I, Afine, fine_diag_pos, I.lmax_bound.p);
  } else {
    if (L.n > 0) SHAKTI_LAUNCH(amg_dinv_kernel, div_up(L.n, 256), 256, 0, s, L.n, fine_diag_pos, Afine.val.p, L.dinv.p);
    if (cheby && L.n > 0)
      SHAKTI_LAUNCH(amg_gershgorin_kernel, bound_blocks(L.n, I.sm_count), 256, 0, s, view(Afine), L.dinv.p,
                    reinterpret_cast<unsigned long long*>(I.lmax_bound.p));
  }
  if (cheby) {
    comm_allreduce_max(I.lmax_bound.p, 1, s);
    launch_cheby_coef(I, 1, true);
  }
  sync_cycle_precision(I, 0, Afine, false, fine);
}

void Amg::refresh(const DevSell& Afine, const int32_t* fine_diag_pos) {
  Impl& I = *p_;
  cudaStream_t s = I.s;
  I.graph_valid = false;
  if (!I.built) { build_hierarchy(I, Afine, fine_diag_pos); I.warm = false; }
  else {
    { SHAKTI_PHASE("rf_numeric", s); for (size_t l = 0; l < I.lv.size(); ++l) numeric_level(I, l, Afine, fine_diag_pos); }
    { SHAKTI_PHASE("rf_tail", s); refresh_tail(I, Afine); }
  }
  bool fine_done;
  { SHAKTI_PHASE("rf_bounds", s); fine_done = update_smoother_bounds(I, Afine, fine_diag_pos); }
  { SHAKTI_PHASE("rf_f32", s); for (size_t l = 0; l < I.lv.size(); ++l) sync_cycle_precision(I, l, Afine, true, fine_done); }
  if (I.dense_coarse) {
    AmgLevel& L = *I.lv.back();
    const DevSell& A = (I.lv.size() == 1) ? Afine : L.A;
    const int32_t N = I.cN, nmax = std::max(I.cnmax, 1);
    SHAKTI_CUDA(cudaMemsetAsync(I.dense_rows.p, 0, sizeof(double) * (size_t)nmax * N, s));
    if (L.n > 0)
      SHAKTI_LAUNCH(amg_dense_rows_kernel, div_up(L.n, 128), 128, 0, s, view(A), A.rowlen.p, I.ccolmap.p, L.n, N, I.dense_rows.p);
    comm_allgather(I.dense_rows.p, I.dense_gather.p, nmax * N, s);
    SHAKTI_CUDA(cudaMemsetAsync(I.dense.p, 0, sizeof(double) * 2 * (size_t)N * N, s));
    SHAKTI_CUDA(cudaMemsetAsync(I.info.p, 0, sizeof(int), s));
    SHAKTI_LAUNCH(amg_dense_assemble_kernel, div_up((int64_t)N * N, 256), 256, 0, s, N, nmax, comm().nranks, I.coff.p,
                  I.dense_gather.p, I.dense.p);
    SHAKTI_LAUNCH(amg_dense_invert_kernel, 1, 1024, N * sizeof(double), s, N, I.dense.p, I.info.p);
  }
  ++refreshes_;
}

// x_is_d: CHEBY_X_IS_D (never on a level that runs on its half-precision copy: see seams_apply, restrict_starts)
template <class T>
static void cheby_step(Amg::Impl& I, const DevSell& A, const T* dinv, const T* b, const T* x, T* d, T* x_out, const double* cf,
                       cudaStream_t s, bool x_is_d = false) {
  if (x_is_d) launch_cheby<T, CHEBY_X_IS_D>(view_as<T>(A), dinv, b, x, d, x_out, cf, s);
  else launch_cheby<T>(view_as<T>(A), dinv, b, x, d, x_out, cf, s);
}
template <>
void cheby_step<float>(Amg::Impl& I, const DevSell& A, const float* dinv, const float* b, const float* x, float* d, float* x_out,
                       const double* cf, cudaStream_t s, bool x_is_d) {
  if (x_is_d)
    launch_cheby<float, CHEBY_X_IS_D>(viewf(A), dinv, b, x, d, x_out, cf, s);
  else if (uses_half(I, A))
    SHAKTI_LAUNCH_PDL(amg_cheby_h_kernel, div_up((int64_t)A.n_slices * 32, 256), 256, 0, s, A.n_rows, A.n_slices, A.slice_ptr.p, A.col.p,
                      A.valh.p, dinv, b, x, d, x_out, cf);
  else
    launch_cheby<float>(viewf(A), dinv, b, x, d, x_out, cf, s);
}
template <class T>
static void level_residual(Amg::Impl& I, const DevSell& A, const T* dinv, const T* x, const T* b, T* r, cudaStream_t s) {
  launch_residual<T>(view_as<T>(A), x, b, r, s);
}
template <>
void level_residual<float>(Amg::Impl& I, const DevSell& A, const float* dinv, const float* x, const float* b, float* r, cudaStream_t s) {
  if (uses_half(I, A))
    SHAKTI_LAUNCH_PDL(amg_resid_h_kernel, div_up((int64_t)A.n_slices * 32, 256), 256, 0, s, A.n_rows, A.n_slices, A.slice_ptr.p, A.col.p,
                      A.valh.p, dinv, b, x, r);
  else
    launch_residual<float>(viewf(A), x, b, r, s);
}

// `sweeps` smoothing steps on A x = b, in place on v.x (ping-pong with v.x2).  zero_guess: v.x is
// taken as 0 and the first step needs no SpMV.  Every SpMV is preceded by the level's halo exchange
// unless the caller says the ghosts are already current.  seam (Chebyshev on the fine level, see
// seams_apply): kSeamEntry -- the zero-guess step was done by amg_cycle_entry_kernel, which left d
// unwritten; kSeamExit -- the last sweep is left to Amg::apply, which reads I.exit_x.
enum { kSeamEntry = 1, kSeamExit = 2 };
template <class T>
static void smooth(Amg::Impl& I, AmgLevel& L, const DevSell& A, const T* b, int sweeps, bool zero_guess, bool ghosts_current,
                   int seam = 0) {
  cudaStream_t s = I.s;
  CycleVecs<T>& v = vecs<T>(L);
  if (sweeps <= 0) {
    if (zero_guess) launch_fill_t<T>(L.n, (T)0, v.x.p, s);
    return;
  }
  if (I.opt.smoother == 1) {   // Chebyshev polynomial of degree `sweeps` on D^-1 A, interval [lmax/ratio, lmax]
    // coefficients: amg_cheby_coef_kernel
    SHAKTI_REQUIRE(sweeps <= I.coef_sweeps, "AMG: more Chebyshev sweeps than coefficients");
    const double* cf = I.coef.p + (size_t)L.index * I.coef_stride;
    int k0 = 0;
    if (zero_guess) {
      if (L.n && !(seam & kSeamEntry))
        SHAKTI_LAUNCH_PDL((amg_cheby_first_kernel<T>), div_up(L.n, 256), 256, 0, s, L.n, v.dinv.p, b, cf, v.d.p, v.x.p);
      k0 = 1;
    }
    for (int k = k0; k < sweeps; ++k) {
      if (I.opt.smoother_halo && !(ghosts_current && k == k0)) L.halo->exchange(v.x.p, s);
      if ((seam & kSeamExit) && k == sweeps - 1) {
        I.exit_x = reinterpret_cast<const float*>(v.x.p);
        break;
      }
      if (L.n) cheby_step<T>(I, A, v.dinv.p, b, v.x.p, v.d.p, v.x2.p, cf + 2 + 2 * k, s, (seam & kSeamEntry) && k == k0);
      std::swap(v.x.p, v.x2.p);
    }
  } else {                      // damped Jacobi
    const double om = I.opt.smoother_omega;
    int k0 = 0;
    if (zero_guess) { launch_scaled_mul<T>(L.n, v.dinv.p, b, om, v.x.p, s); k0 = 1; }
    for (int k = k0; k < sweeps; ++k) {
      if (I.opt.smoother_halo && !(ghosts_current && k == k0)) L.halo->exchange(v.x.p, s);
      launch_jacobi<T>(view_as<T>(A), v.dinv.p, b, v.x.p, v.x2.p, om, s);
      std::swap(v.x.p, v.x2.p);
    }
  }
}

// Does the restriction onto level c also take c's first smoothing step (launch_restrict_cheby_first)?  For a
// level smoothed locally by Chebyshev from a zero guess, with a second step to take over the fused start's
// unwritten d: not the replicated level, not the coarsest level, not a level on its half-precision copy.
static bool restrict_starts(const Amg::Impl& I, size_t c) {
  const AmgLevel& C = *I.lv[c];
  return I.opt.smoother == 1 && I.opt.presmooth >= 2 && !C.last && (int)c != I.tail_level && !uses_half(I, C.A);
}

template <class T>
static void vcycle(Amg::Impl& I, const DevSell& Afine, bool seams) {
  cudaStream_t s = I.s;
  const int nl = (int)I.lv.size();
  for (int l = 0; l < nl; ++l) {   // downward; level l's right-hand side is vecs(l).b
    AmgLevel& L = *I.lv[l];
    CycleVecs<T>& v = vecs<T>(L);
    const DevSell& A = (l == 0) ? Afine : L.A;
    if (l == I.tail_level) {
      // replicated part: all-gather this level's right-hand side, solve on every rank, pick own + ghost entries
      T* tb = I.tail->rhs_buffer<T>();
      if (comm().p2p) {
        I.tail_gather.allgatherv<T, T>(v.b.p, tb, s);
      } else {
        SHAKTI_CUDA(cudaMemsetAsync(I.tail_rhs_d.p, 0, sizeof(double) * I.tail_nmax, s));
        if (L.n) SHAKTI_LAUNCH((amg_convert_kernel<T, double>), div_up(L.n, 256), 256, 0, s, L.n, v.b.p, I.tail_rhs_d.p);
        comm_allgather(I.tail_rhs_d.p, I.tail_gather_d.p, I.tail_nmax, s);
        SHAKTI_LAUNCH((amg_compact_kernel<T>), div_up(I.tail_N, 128), 128, 0, s, I.tail_N, I.tail_nmax, comm().nranks, I.tail_off.p,
                      I.tail_gather_d.p, tb);
      }
      const T* tx;
      {
        CommSerialScope serial;
        tx = I.tail->cycle<T>(I.tailM);
      }
      if (L.n_cols) SHAKTI_LAUNCH_PDL((amg_gather_map_kernel<T>), div_up(L.n_cols, 256), 256, 0, s, L.n_cols, I.tail_gid.p, tx, v.x.p);
      break;
    }
    if (L.last) {
      if (I.dense_coarse) {
        const int32_t N = I.cN, nmax = std::max(I.cnmax, 1);
        if (comm().active()) {
          SHAKTI_CUDA(cudaMemsetAsync(I.crhs.p, 0, sizeof(double) * nmax, s));
          if (L.n) SHAKTI_LAUNCH((amg_convert_kernel<T, double>), div_up(L.n, 256), 256, 0, s, L.n, v.b.p, I.crhs.p);
          comm_allgather(I.crhs.p, I.cgather.p, nmax, s);
          SHAKTI_LAUNCH((amg_compact_kernel<double>), div_up(N, 128), 128, 0, s, N, nmax, comm().nranks, I.coff.p, I.cgather.p, I.cglob.p);
          SHAKTI_LAUNCH((amg_dense_apply_kernel<double, double>), div_up((int64_t)N * 32, 128), 128, 0, s, N, I.dense.p, I.cglob.p, I.csol.p);
          if (L.n) SHAKTI_LAUNCH((amg_convert_kernel<double, T>), div_up(L.n, 256), 256, 0, s, L.n, I.csol.p + I.coff_me, v.x.p);
        } else if (L.n) {
          SHAKTI_LAUNCH_PDL((amg_dense_apply_kernel<T, T>), div_up((int64_t)L.n * 32, 128), 128, 0, s, L.n, I.dense.p, v.b.p, v.x.p);
        }
      } else {
        smooth<T>(I, L, A, v.b.p, 8, true, false);
      }
      break;
    }
    const bool started = l > 0 && restrict_starts(I, l);
    smooth<T>(I, L, A, v.b.p, I.opt.presmooth, true, false, (seams && l == 0) || started ? kSeamEntry : 0);
    L.halo->exchange(v.x.p, s);
    level_residual<T>(I, A, v.dinv.p, v.x.p, v.b.p, v.r.p, s);
    CycleVecs<T>& vc = vecs<T>(*I.lv[l + 1]);
    if (restrict_starts(I, l + 1))
      launch_restrict_cheby_first<T>(view_as<T>(L.R), v.r.p, vc.dinv.p, I.coef.p + (size_t)(l + 1) * I.coef_stride, vc.b.p, vc.x.p, s);
    else
      launch_spmv<T>(view_as<T>(L.R), v.r.p, vc.b.p, s);
  }
  for (int l = nl - 2; l >= 0; --l) {   // upward
    AmgLevel& L = *I.lv[l];
    CycleVecs<T>& v = vecs<T>(L);
    const DevSell& A = (l == 0) ? Afine : L.A;
    AmgLevel& C = *I.lv[l + 1];
    if (l + 1 != I.tail_level) C.halo->exchange(vecs<T>(C).x.p, s);   // the replicated level's ghosts are already set
    // own rows AND ghost rows of P are applied: the ghost part of x stays consistent with its owner
    // (it was exchanged before the residual), so the first post-smoothing step needs no exchange
    launch_spmv_add<T>(view_as<T>(L.P), vecs<T>(C).x.p, v.x.p, s);
    smooth<T>(I, L, A, v.b.p, I.opt.postsmooth, false, true, seams && l == 0 ? kSeamExit : 0);
  }
}

// Runs the V-cycle, through a captured CUDA graph when enabled.  The ping-pong pointers are put
// back after every cycle, so each cycle (and each capture) uses the same buffers in the same roles
// and a re-capture after a refresh only updates kernel arguments (cudaGraphExecUpdate).
template <class T>
static void run_cycle(Amg::Impl& I, const DevSell& Afine, bool seams = false) {
  cudaStream_t s = I.s;
  std::vector<std::pair<T*, T*>> saved;
  for (auto& L : I.lv) saved.push_back({vecs<T>(*L).x.p, vecs<T>(*L).x2.p});
  auto restore = [&]() {
    I.result_ptr = vecs<T>(*I.lv[0]).x.p;
    for (size_t l = 0; l < I.lv.size(); ++l) { vecs<T>(*I.lv[l]).x.p = saved[l].first; vecs<T>(*I.lv[l]).x2.p = saved[l].second; }
  };
  if (!I.opt.cuda_graph || !I.warm) {
    vcycle<T>(I, Afine, seams);
    restore();
    I.warm = true;
    return;
  }
  const void* key[5] = {Afine.slice_ptr.p, Afine.col.p, Afine.val.p, Afine.valf.p, Afine.valh.p};
  if (!std::equal(key, key + 5, I.graph_key) || seams != I.graph_seams) I.graph_valid = false;
  if (!I.graph_valid) {
    std::copy(key, key + 5, I.graph_key);
    I.graph_seams = seams;
    const int64_t before = g_kernel_launches;
    SHAKTI_CUDA(cudaStreamBeginCapture(s, cudaStreamCaptureModeRelaxed));
    cudaGraph_t graph = nullptr;
    try {
      vcycle<T>(I, Afine, seams);
    } catch (...) {
      cudaStreamEndCapture(s, &graph);
      if (graph) cudaGraphDestroy(graph);
      restore();
      throw;
    }
    SHAKTI_CUDA(cudaStreamEndCapture(s, &graph));
    restore();
    I.graph_launches = g_kernel_launches - before;
    g_kernel_launches = before;     // captured, not executed
    bool updated = false;
    if (I.gexec) {
      cudaGraphExecUpdateResultInfo info;
      updated = cudaGraphExecUpdate(I.gexec, graph, &info) == cudaSuccess;
      if (!updated) { cudaGetLastError(); cudaGraphExecDestroy(I.gexec); I.gexec = nullptr; }
    }
    if (!updated) SHAKTI_CUDA(cudaGraphInstantiate(&I.gexec, graph, 0));
    SHAKTI_CUDA(cudaGraphDestroy(graph));
    I.graph_valid = true;
  }
  SHAKTI_CUDA(cudaGraphLaunch(I.gexec, s));
  g_kernel_launches += I.graph_launches;
}

bool Amg::launch_level_smoother(int level, const DevSell& Afine, int64_t* rows, int64_t* nnz, int* value_bytes) {
  Impl& I = *p_;
  if (!I.built || level < 0 || level >= (int)I.lv.size()) return false;
  AmgLevel& L = *I.lv[level];
  const DevSell& A = (level == 0) ? Afine : L.A;
  if (rows) *rows = L.n;
  if (nnz) *nnz = A.nnz;
  if (value_bytes) *value_bytes = uses_half(I, A) ? 2 : (I.opt.fp32_cycle ? 4 : 8);
  if (L.n == 0) return true;
  if (I.opt.fp32_cycle) cheby_step<float>(I, A, L.vf.dinv.p, L.vf.b.p, L.vf.x.p, L.vf.d.p, L.vf.x2.p, I.fixed_coef.p, I.s);
  else launch_cheby<double>(view(A), L.vd.dinv.p, L.vd.b.p, L.vd.x.p, L.vd.d.p, L.vd.x2.p, I.fixed_coef.p, I.s);
  return true;
}

template <class T>
static void level_kernel(Amg::Impl& I, int l, int which, const DevSell& A) {
  AmgLevel& L = *I.lv[l];
  CycleVecs<T>& v = vecs<T>(L);
  CycleVecs<T>& vc = vecs<T>(*I.lv[l + (which == 1 ? 0 : 1)]);
  if (which == 1) level_residual<T>(I, A, v.dinv.p, v.x.p, v.b.p, v.r.p, I.s);
  else if (which == 3) launch_spmv_add<T>(view_as<T>(L.P), vc.x.p, v.x.p, I.s);
  else if (restrict_starts(I, l + 1))
    launch_restrict_cheby_first<T>(view_as<T>(L.R), v.r.p, vc.dinv.p, I.coef.p + (size_t)(l + 1) * I.coef_stride, vc.b.p, vc.x.p, I.s);
  else
    launch_spmv<T>(view_as<T>(L.R), v.r.p, vc.b.p, I.s);
}
bool Amg::launch_level_kernel(int level, int which, const DevSell& Afine, int64_t info[7]) {
  Impl& I = *p_;
  if (!I.built || level < 0 || level >= (int)I.lv.size() || which < 0 || which > 3) return false;
  AmgLevel& L = *I.lv[level];
  const DevSell& A = (level == 0) ? Afine : L.A;
  // the cycle restricts and prolongs only between levels it runs on this rank
  const bool transfer = !L.last && level + 1 < (int)I.lv.size() && (I.tail_level < 0 || level < I.tail_level);
  if (which >= 2 && !transfer) return false;
  const DevSell& M = which == 2 ? L.R : which == 3 ? L.P : A;
  info[0] = M.n_rows; info[1] = M.n_cols; info[2] = M.nnz; info[3] = M.max_width;
  info[4] = &M == &A && uses_half(I, A) ? 2 : (I.opt.fp32_cycle ? 4 : 8);   // R and P have no half-precision copy
  info[5] = I.opt.fp32_cycle ? 4 : 8;
  info[6] = which == 2 && restrict_starts(I, level + 1);
  if (which == 0) return launch_level_smoother(level, Afine, nullptr, nullptr);
  if (M.n_rows == 0) return true;
  if (I.opt.fp32_cycle) level_kernel<float>(I, level, which, A);
  else level_kernel<double>(I, level, which, A);
  return true;
}

template <class T> T* Amg::rhs_buffer() { return vecs<T>(*p_->lv[0]).b.p; }
template <class T> const T* Amg::cycle(const DevSell& Afine) {
  run_cycle<T>(*p_, Afine);
  return static_cast<const T*>(p_->result_ptr);
}
template float* Amg::rhs_buffer<float>();
template double* Amg::rhs_buffer<double>();
template const float* Amg::cycle<float>(const DevSell&);
template const double* Amg::cycle<double>(const DevSell&);

// Do the cycle's seams with the Krylov vectors fuse into the fine level's first and last smoothing steps?
// That takes the mixed-precision cycle with Chebyshev smoothing of the fine level on its fp32 copy, a first
// step followed by at least one more (the fused start leaves d unwritten) and at least one post-smoothing step.
static bool seams_apply(const Amg::Impl& I, const DevSell& Afine) {
  const AmgLevel& L0 = *I.lv[0];
  return I.opt.fp32_cycle && I.opt.smoother == 1 && I.opt.presmooth >= 2 && I.opt.postsmooth >= 1 && !L0.last &&
         I.tail_level != 0 && L0.n > 0 && !uses_half(I, Afine);
}

void Amg::apply(const DevSell& Afine, const double* rin, double* z) {
  Impl& I = *p_;
  cudaStream_t s = I.s;
  AmgLevel& L0 = *I.lv[0];
  if (seams_apply(I, Afine)) {
    // entry and exit read and write the Krylov vectors, which change every iteration: launched outside the graph
    SHAKTI_LAUNCH(amg_cycle_entry_kernel, div_up(L0.n, 256), 256, 0, s, L0.n, rin, L0.vf.dinv.p, I.coef.p, L0.vf.b.p, L0.vf.x.p);
    run_cycle<float>(I, Afine, true);
    const double* cf = I.coef.p + 2 + 2 * (I.opt.postsmooth - 1);
    const SellViewT<float> A = viewf(Afine);
    if (A.n_rows < kChebyWideRowsBelow)
      SHAKTI_LAUNCH((amg_cheby_kernel<float, 8, CHEBY_EXIT>), A.n_slices, 256, 0, s, A, L0.vf.dinv.p, L0.vf.b.p, I.exit_x, L0.vf.d.p,
                    nullptr, cf, z);
    else
      sell_row_bound_dispatch<float>(A.max_width, [&](auto rb) {
        SHAKTI_LAUNCH((amg_cheby_kernel<float, 1, CHEBY_EXIT, rb.value>), div_up((int64_t)A.n_slices * 32, 256), 256, 0, s, A,
                      L0.vf.dinv.p, L0.vf.b.p, I.exit_x, L0.vf.d.p, nullptr, cf, z);
      });
  } else if (I.opt.fp32_cycle) {
    launch_d2f(L0.n, rin, L0.vf.b.p, s);
    run_cycle<float>(I, Afine);
    launch_f2d(L0.n, static_cast<const float*>(I.result_ptr), z, s);
  } else {
    if (L0.n) SHAKTI_CUDA(cudaMemcpyAsync(L0.vd.b.p, rin, sizeof(double) * L0.n, cudaMemcpyDeviceToDevice, s));
    run_cycle<double>(I, Afine);
    if (L0.n) SHAKTI_CUDA(cudaMemcpyAsync(z, I.result_ptr, sizeof(double) * L0.n, cudaMemcpyDeviceToDevice, s));
  }
}

}  // namespace shakti

// ---------------------------------------------------------------- host-only test hook
// Strength filter + greedy aggregation of a square CSR matrix, exactly as coarsen_level() does on one rank.
extern "C" int shakti_host_amg_aggregate(int32_t n, const int32_t* rowptr, const int32_t* col, const double* val,
                                         double theta, const uint8_t* exclude, int32_t* agg_out, int32_t* n_agg) {
  try {
    if (n <= 0 || !rowptr || !col || !agg_out || !n_agg) throw shakti::Error(SHAKTI_ERR_INVALID, "bad arguments");
    shakti::HostCsr A;
    A.n_rows = A.n_cols = n;
    A.rowptr.assign(rowptr, rowptr + n + 1);
    A.col.assign(col, col + rowptr[n]);
    std::vector<uint8_t> excl;
    if (exclude) excl.assign(exclude, exclude + n);
    std::vector<uint8_t> strong;
    if (theta > 0 && val) {
      std::vector<double> diag(n, 0.0);
      for (int32_t i = 0; i < n; ++i)
        for (int32_t k = rowptr[i]; k < rowptr[i + 1]; ++k)
          if (col[k] == i) diag[i] = std::fabs(val[k]);
      strong.assign(A.nnz(), 0);
      for (int32_t i = 0; i < n; ++i)
        for (int32_t k = rowptr[i]; k < rowptr[i + 1]; ++k) {
          const int32_t j = col[k];
          if (j == i) continue;
          const double a = std::fabs(val[k]);
          strong[k] = (a >= theta * std::sqrt(diag[i] * diag[j])) && a > 0;
        }
    }
    std::vector<int32_t> agg;
    *n_agg = shakti::aggregate(A, n, excl, strong, agg);
    std::copy(agg.begin(), agg.end(), agg_out);
    return SHAKTI_OK;
  } catch (const std::exception& e) {
    shakti::set_last_error(e.what());
    return SHAKTI_ERR_INVALID;
  }
}

