// Device-side data structures and kernel launch wrappers.
#pragma once
#include <cuda_fp16.h>

#include "common.h"
#include "moulin.h"
#include "prep.h"
#include "sell_row.h"

namespace shakti {

// constants of source/params.py:4-11 plus derived values, passed to kernels by value
struct DevParams {
  double g, rho_i, rho_w, nu, Lh, omega, n, A;
  double cm;    // 1/rho_i - 1/rho_w
  double rwg;   // rho_w * g
  double inv_rwg, inv_Lh, cm_over_Lh;   // reciprocals, so the cell kernels do not divide by constants
  int n_is_3;   // Glen exponent is exactly 3 => closure terms are polynomials
};

DevParams make_dev_params(const shakti_params& p);

// SELL-32 sparse matrix on the device (layout: prep.h HostSell)
struct DevSell {
  int32_t n_rows = 0, n_cols = 0, n_slices = 0;
  int32_t max_width = 0;        // longest row
  int64_t padded = 0, nnz = 0;
  DevBuf<int32_t> slice_ptr, col, rowlen;
  DevBuf<double> val;
  mutable DevBuf<float> valf;   // single-precision copy of val (mixed-precision AMG cycle), made on demand
  mutable DevBuf<__half> valh;  // half-precision copy of D^-1 A (smoother / residual of the large AMG levels)
  void upload_pattern(const HostSell& h, int64_t nnz_);
  void refresh_f32(cudaStream_t s) const;   // valf <- val
  // valh <- dinv[row] * val: the row-scaled operator has a unit diagonal and off-diagonals of order 1, which is
  // what makes 16-bit storage possible (raw Jacobian entries span 1e-11 ... 4e-3)
  void refresh_f16_scaled(const double* dinv, cudaStream_t s) const;
};

template <class T>
struct SellViewT {
  int32_t n_rows, n_slices;
  const int32_t* slice_ptr;
  const int32_t* col;
  const T* val;
  int32_t max_width;   // longest row: picks the row bound of the one-thread-per-row kernels (sell_row.h)
};
using SellView = SellViewT<double>;
inline SellView view(const DevSell& a) { return {a.n_rows, a.n_slices, a.slice_ptr.p, a.col.p, a.val.p, a.max_width}; }
inline SellViewT<float> viewf(const DevSell& a) { return {a.n_rows, a.n_slices, a.slice_ptr.p, a.col.p, a.valf.p, a.max_width}; }
template <class T> inline SellViewT<T> view_as(const DevSell& a);
template <> inline SellViewT<double> view_as<double>(const DevSell& a) { return view(a); }
template <> inline SellViewT<float> view_as<float>(const DevSell& a) { return viewf(a); }

// Pointers of the vertex fields the element kernels read (all n_local long)
struct FieldPtrs {
  const double *x, *y, *h0, *N, *N_n, *b, *qx, *qy, *G, *melt, *storage, *inputs;
  const uint8_t* isbc;
};

// ---- quadrature tables in __constant__ memory
void upload_k_rule(int n, const double* pts_xy, const double* wts, cudaStream_t s);       // for Kbar
void upload_reaction_rule(int n, const double* pts_xy, const double* wts, cudaStream_t s); // closure/storage

// ---- element kernels
void launch_kbar(int32_t ne, const int32_t* c0, const int32_t* c1, const int32_t* c2,
                 const double* x, const double* y, const double* b, const double* qx,
                 const double* qy, double* kbar, DevParams p, cudaStream_t s);
void launch_assemble_atomic(int32_t ne, int32_t n_owned, const int32_t* c0, const int32_t* c1,
                            const int32_t* c2, const int32_t* slot, FieldPtrs f, const double* kbar,
                            double dt, double N_bdry, double* F, double* Jval, int want_J,
                            DevParams p, cudaStream_t s);
struct AssemblyPlanView {   // device arrays of prep.h AssemblyBlocks
  int32_t n_owned, rows_per_block, n_blocks, cap, vcap;
  const int32_t *blk_eptr, *blk_elems;
  const uint16_t* blk_lv;
  const int32_t *blk_hptr, *blk_halo, *inc_ptr;
  const uint16_t* inc_code;
  const uint32_t* src;
};
void launch_assemble_blocks(const AssemblyPlanView& plan, FieldPtrs f, const double* kbar, double dt, double N_bdry,
                            const int32_t* slice_ptr, double* F, double* Jval, int want_J, DevParams p, cudaStream_t s);
void launch_apply_bc(int32_t n_owned, const uint8_t* isbc, const double* N, double N_bdry,
                     const int32_t* diag_pos, double* F, double* Jval, int want_J, cudaStream_t s);

// ---- water-budget diagnostics (shakti_diagnostics, shakti_record_diagnostics)
// Rank-local values before the global reduction: kDiagSums sums (all-reduced by sum), then maxima (by max;
// the minimum of N is carried as the maximum of -N).
enum {
  kDiagArea = 0, kDiagVolume, kDiagInput, kDiagMelt, kDiagClosure, kDiagStorage, kDiagOutflow, kDiagImbalance, kDiagIntN,
  kDiagSums,
  kDiagNegNmin = kDiagSums, kDiagNmax, kDiagBmax,
  kDiagVals
};
// blocks of the cell pass (= partials it writes)
int diagnostics_parts(int32_t ne, int sm_count);
// counted: 1 for the local cells this rank adds (prep.h HostMesh::cell_counted); partial: nparts x kDiagVals scratch.
// Writes the rank's values to vals[kDiagVals] and, if row != NULL, the finished record (one rank only).
void launch_diagnostics(int32_t ne, const int32_t* c0, const int32_t* c1, const int32_t* c2, const uint8_t* counted, FieldPtrs f,
                        const double* kbar, double dt, DevParams p, int nparts, double* partial, double* vals, double* row,
                        double its, double residual, cudaStream_t s);
// record row from globally reduced vals (several ranks)
void launch_diagnostics_row(const double* vals, double* row, double dt, double its, double residual, cudaStream_t s);
// rank values: input += q, imbalance -= q (q: discharge of this rank's moulins)
void launch_diagnostics_moulins(double* vals, double q, cudaStream_t s);

// ---- moulins (shakti_set_moulins): this rank's moulin rows, each with its moulins in caller order
struct MoulinView {
  int32_t n_rows;
  const int32_t* row;    // n_rows local row ids (owned), ascending
  const int32_t* rptr;   // n_rows + 1: moulins of row r are rptr[r] .. rptr[r+1]-1
  const int64_t* kptr;   // moulins + 1: knots of moulin k are kptr[k] .. kptr[k+1]-1 of tk, qk
  const double *tk, *qk;
  double period;
};
// F[row] -= sum over the row's moulins of Q_k(t)   (moulin.h hydrograph_at)
void launch_moulin_source(const MoulinView& mv, double t, double* F, cudaStream_t s);

// ---- nodal updates (solvers.py:186-197)
void launch_update_q(int32_t n_owned, const int32_t* win, const double* x, const double* y,
                     const double* h0, const double* N, const double* b, double* qx, double* qy,
                     DevParams p, cudaStream_t s);
void launch_update_melt(int32_t n_owned, const int32_t* win, const double* x, const double* y,
                        const double* h0, const double* N, const double* b, const double* qx,
                        const double* qy, const double* G, const double* melt_old, double* melt_new,
                        DevParams p, cudaStream_t s);
// q and melt_n in one pass (same results as launch_update_q followed by launch_update_melt)
void launch_update_q_melt(int32_t n_owned, const int32_t* win, const double* x, const double* y,
                          const double* h0, const double* N, const double* b, double* qx, double* qy,
                          const double* G, const double* melt_old, double* melt_new, DevParams p, cudaStream_t s);
void launch_update_b(int32_t n_owned, const int32_t* win, const double* x, const double* y,
                     const double* h0, const double* N, const double* b_old, const double* qx,
                     const double* qy, const double* G, const double* melt, double* b_new, double dt,
                     double b_min, DevParams p, cudaStream_t s);

// ---- sparse / vector kernels (T = double, or float for the mixed-precision AMG cycle)
template <class T> void launch_spmv(SellViewT<T> A, const T* x, T* y, cudaStream_t s);                 // y = A x
template <class T> void launch_residual(SellViewT<T> A, const T* x, const T* b, T* r, cudaStream_t s); // r = b - A x
// x_out = x + omega * dinv .* (b - A x)
template <class T> void launch_jacobi(SellViewT<T> A, const T* dinv, const T* b, const T* x, T* x_out, double omega, cudaStream_t s);
template <class T> void launch_spmv_add(SellViewT<T> A, const T* x, T* y, cudaStream_t s);             // y += A x
// b_c = R r and the first Chebyshev step from a zero guess on the coarse level, x_c = dinv_c b_c inv_theta[0]
template <class T>
void launch_restrict_cheby_first(SellViewT<T> R, const T* r, const T* dinv_c, const double* inv_theta, T* b_c, T* x_c, cudaStream_t s);
template <class T> void launch_scaled_mul(int64_t n, const T* a, const T* b, double scale, T* out, cudaStream_t s);  // out = scale a.*b
template <class T> void launch_fill_t(int64_t n, T v, T* x, cudaStream_t s);
void launch_d2f(int64_t n, const double* a, float* out, cudaStream_t s);
void launch_f2d(int64_t n, const float* a, double* out, cudaStream_t s);
void launch_extract_dinv(int32_t n, const int32_t* diag_pos, const double* val, double* dinv, cudaStream_t s);

// reductions: out[k] = <V_k, w>, V_k = V + k*ld, k < nvec; result in device memory `out`
struct Reducer {
  DevBuf<double> partial;
  DevBuf<unsigned int> counter;
  int max_blocks = 0;
  void init(int sm_count);
};
void launch_multi_dot(Reducer& red, int64_t n, int nvec, const double* V, int64_t ld, const double* w,
                      double* out, cudaStream_t s);
// w -= sum_k h[k] V_k   (h on device)
void launch_multi_axpy_neg(int64_t n, int nvec, const double* V, int64_t ld, const double* h, double* w,
                           cudaStream_t s);
// fused: w -= V h; out[0..nvec) = V^T w_new; out[nvec] = <w_new,w_new>.  false: nvec too large, nothing done
bool launch_orth_update_dot(Reducer& red, int64_t n, int nvec, const double* V, int64_t ld, const double* h, double* w,
                            double* out, cudaStream_t s);
void launch_multi_axpy_neg_scale(int64_t n, int nvec, const double* V, int64_t ld, const double* h, double* w, double scale,
                                 cudaStream_t s);
// y = sum_k h[k] V_k
void launch_combine(int64_t n, int nvec, const double* V, int64_t ld, const double* h, double* y,
                    cudaStream_t s);
// dst_host[0..count) = src[0..count): a KERNEL stores into page-locked host memory (cudaMallocHost memory is
// device-accessible under unified addressing).  The small per-iteration reads of the solvers must not go
// through the copy engines: while the asynchronous save path moves hundreds of MB to the host, an 8-byte
// cudaMemcpyAsync would queue behind a 128 MB chunk (measured: 16 ms per step lost at C4).  The caller
// synchronises the stream before reading.
void launch_readback(const double* src, double* dst_host, int count, cudaStream_t s);
void launch_axpy(int64_t n, double alpha, const double* x, double* y, cudaStream_t s);  // y += alpha x
void launch_xmy_masked(int64_t n, const double* a, const uint8_t* mask, double* out, cudaStream_t s);
void launch_gather(int64_t n, const int32_t* idx, const double* src, double* dst, cudaStream_t s);   // dst[i] = src[idx[i]]
void launch_scatter(int64_t n, const int32_t* idx, const double* src, double* dst, cudaStream_t s);  // dst[idx[i]] = src[i]
// model_setup data ingestion on the device (reference model_setup.py:68-91)
void launch_interp_grid(int64_t n, const double* px, const double* py, int nx, int ny, const double* xg, const double* yg,
                        const double* f, double* out, cudaStream_t s);
void launch_points_in_polygon(int64_t n, const double* px, const double* py, int m, const double* poly_xy, double* out,
                              cudaStream_t s);
void launch_head0(int64_t n, const double* z_b, const double* z_s, double ratio, double* h0, cudaStream_t s);
void launch_interleave(int64_t n, const double* a, const double* b, double* ab, cudaStream_t s);
void launch_deinterleave(int64_t n, const double* ab, double* a, double* b, cudaStream_t s);

}  // namespace shakti
