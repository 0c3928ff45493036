// Bitwise check of the SELL-32 row product (shakti-fenics_b200/csrc/sell_row.h): on random slices of every width
// 0 ... 8, with rows shorter than their slice padded as the library pads them (value 0, column of the row itself),
// the load-before-gather path (RB = 8) must give the same bits as the plain loop (RB = 0), and both the same bits as
// a host chain of fmaf from 0 in entry order.  Built and run by tests/test_gpu_sell_kernels.py; prints "ok" or the
// first mismatches and exits non-zero.
#include <cmath>
#include <cstdio>
#include <cstring>
#include <random>
#include <vector>

#include "sell_row.h"

using shakti::sell_row_product;

template <int RB>
__global__ void row_products(int n_slices, const int32_t* slice_ptr, const int32_t* col, const float* val, const float* x,
                             float* y) {
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  const int slice = row >> 5;
  if (slice >= n_slices) return;
  const int32_t base = slice_ptr[slice];
  const int32_t w = (slice_ptr[slice + 1] - base) >> 5;
  y[row] = sell_row_product<RB>(col + base + (row & 31), val + base + (row & 31), w, x);
}

#define CHECK(e)                                                                        \
  do {                                                                                  \
    cudaError_t err_ = (e);                                                             \
    if (err_ != cudaSuccess) {                                                          \
      std::printf("CUDA error %s at line %d\n", cudaGetErrorString(err_), __LINE__);    \
      return 2;                                                                         \
    }                                                                                   \
  } while (0)

int main() {
  const int n_slices = 9 * 4096, n = 32 * n_slices;
  std::mt19937 rng(12345);
  std::uniform_int_distribution<int> any_col(0, n - 1);
  std::uniform_real_distribution<float> u(-1.f, 1.f);
  std::vector<int32_t> slice_ptr(n_slices + 1, 0), rowlen(n);
  for (int s = 0; s < n_slices; ++s) {
    const int w = s % 9;                                   // every width 0 ... 8
    for (int l = 0; l < 32; ++l) rowlen[32 * s + l] = w == 0 ? 0 : 1 + (int)(rng() % w);
    rowlen[32 * s + (int)(rng() % 32)] = w;                 // one row sets the slice width
    slice_ptr[s + 1] = slice_ptr[s] + 32 * w;
  }
  std::vector<int32_t> col(slice_ptr[n_slices]);
  std::vector<float> val(slice_ptr[n_slices]), x(n);
  for (int s = 0; s < n_slices; ++s) {
    const int w = (slice_ptr[s + 1] - slice_ptr[s]) / 32;
    for (int l = 0; l < 32; ++l)
      for (int k = 0; k < w; ++k) {
        const int r = 32 * s + l, p = slice_ptr[s] + 32 * k + l;
        const bool real = k < rowlen[r];
        col[p] = real ? any_col(rng) : r;
        val[p] = real ? u(rng) * std::ldexp(1.f, (int)(rng() % 40) - 20) : 0.f;
      }
  }
  for (auto& v : x) v = u(rng) * std::ldexp(1.f, (int)(rng() % 40) - 20);
  std::vector<float> ref(n);
  for (int r = 0; r < n; ++r) {
    const int s = r >> 5, w = (slice_ptr[s + 1] - slice_ptr[s]) / 32;
    float acc = 0.f;
    for (int k = 0; k < w; ++k) {
      const int p = slice_ptr[s] + 32 * k + (r & 31);
      acc = std::fmaf(val[p], x[col[p]], acc);
    }
    ref[r] = acc;
  }
  int32_t *d_sp, *d_col;
  float *d_val, *d_x, *d_y0, *d_y8;
  CHECK(cudaMalloc(&d_sp, sizeof(int32_t) * slice_ptr.size()));
  CHECK(cudaMalloc(&d_col, sizeof(int32_t) * col.size()));
  CHECK(cudaMalloc(&d_val, sizeof(float) * val.size()));
  CHECK(cudaMalloc(&d_x, sizeof(float) * n));
  CHECK(cudaMalloc(&d_y0, sizeof(float) * n));
  CHECK(cudaMalloc(&d_y8, sizeof(float) * n));
  CHECK(cudaMemcpy(d_sp, slice_ptr.data(), sizeof(int32_t) * slice_ptr.size(), cudaMemcpyHostToDevice));
  CHECK(cudaMemcpy(d_col, col.data(), sizeof(int32_t) * col.size(), cudaMemcpyHostToDevice));
  CHECK(cudaMemcpy(d_val, val.data(), sizeof(float) * val.size(), cudaMemcpyHostToDevice));
  CHECK(cudaMemcpy(d_x, x.data(), sizeof(float) * n, cudaMemcpyHostToDevice));
  row_products<0><<<n / 256, 256>>>(n_slices, d_sp, d_col, d_val, d_x, d_y0);
  row_products<8><<<n / 256, 256>>>(n_slices, d_sp, d_col, d_val, d_x, d_y8);
  CHECK(cudaGetLastError());
  std::vector<float> y0(n), y8(n);
  CHECK(cudaMemcpy(y0.data(), d_y0, sizeof(float) * n, cudaMemcpyDeviceToHost));
  CHECK(cudaMemcpy(y8.data(), d_y8, sizeof(float) * n, cudaMemcpyDeviceToHost));
  int bad = 0;
  for (int r = 0; r < n; ++r)
    if (std::memcmp(&y0[r], &ref[r], 4) || std::memcmp(&y8[r], &ref[r], 4)) {
      if (bad++ < 10) std::printf("row %d (width %d): host %a, RB=0 %a, RB=8 %a\n", r, rowlen[r], ref[r], y0[r], y8[r]);
    }
  cudaFree(d_sp); cudaFree(d_col); cudaFree(d_val); cudaFree(d_x); cudaFree(d_y0); cudaFree(d_y8);
  if (bad) {
    std::printf("%d of %d rows differ\n", bad, n);
    return 1;
  }
  std::printf("ok: %d rows, slice widths 0-8\n", n);
  return 0;
}
