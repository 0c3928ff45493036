// Smoothed-aggregation algebraic multigrid preconditioner.
//
// The reference solves each Newton system with a sparse direct LU (PETSc preonly+lu behind
// DOLFINx NewtonSolver, solvers.py:52,179), which does not scale to 16M dofs on a GPU; this
// is the B200-native replacement: a hierarchy whose sparsity is fixed by the mesh (symbolic
// phase once, on the host) and whose numbers are recomputed on the device by bandwidth-bound
// kernels whenever the Jacobian changes (prolongator smoothing + two numeric SpGEMMs per level).
#pragma once
#include <memory>

#include "device.h"

namespace shakti {

struct AmgOptions {
  int max_levels = 12;
  int coarse_size = 128;     // dense LU below this many rows
  int presmooth = 1, postsmooth = 1;
  double smoother_omega = 0.67;
  double prolong_omega = 0.67;  // 0 => plain aggregation
  double strength_theta = 0.08; // |a_ij| >= theta 0.5^level sqrt(|a_ii a_jj|) is a strong connection (0: all)
  int smoother = 1;             // 0 damped Jacobi (presmooth/postsmooth sweeps), 1 Chebyshev (degree = sweeps)
  double cheby_ratio = 5.0;     // Chebyshev interval [lmax/ratio, lmax] of D^-1 A
  int fp32_cycle = 1;           // 1: V-cycle in single precision (set-up and Krylov stay fp64)
  int cuda_graph = 1;           // 1: replay the V-cycle as a captured CUDA graph
  int smoother_halo = 1;        // 1: halo exchange before every smoothing step; 0: only before residual / prolongation
                                //    (ghost values lag one step inside the smoother: hybrid smoothing, fewer messages)
  int replicate_below = 100000; // multi-GPU: the first level with at most this many rows in total (and everything below
                                //    it) is replicated on every rank and solved there without communication
};

class Amg {
 public:
  Amg();
  ~Amg();
  // Register the fine pattern (rows x cols, cols >= rows; only the square rows x rows block is
  // coarsened; A and S must outlive this object).  `exclude[i] != 0` rows (Dirichlet) stay out
  // of the coarse space.  The hierarchy itself is built by the first refresh(), level by level:
  // strength of connection needs the values, so host symbolic work and device numerics interleave.
  // `nbrs`/`halo`: halo description and plan of the fine level (empty / unused on one GPU).  On
  // several GPUs the hierarchy is global: aggregates stay inside a rank, P reaches the neighbours'
  // aggregates, R = (P[own rows, own aggregates])^T, every level has its own halo plan, and the
  // coarsest operator is gathered on all ranks.
  void setup(const HostCsr& A, const HostSell& S, const std::vector<uint8_t>& exclude, const std::vector<Neighbor>& nbrs,
             struct HaloPlan* halo, const AmgOptions& opt, int sm_count, cudaStream_t s);
  // Numeric phase: recompute P, R, coarse operators and smoother diagonals from the fine values.
  void refresh(const DevSell& Afine, const int32_t* fine_diag_pos);
  // Per-solve update of the fine-level smoother only (diagonal + safe Chebyshev bound) for
  // solves that reuse a lagged hierarchy.
  void refresh_fine_smoother(const DevSell& Afine, const int32_t* fine_diag_pos);
  // z = M^-1 r : one V-cycle from a zero initial guess.  r: n rows; z: n_cols-long buffer
  // (entries beyond n rows are left untouched and must be zero / halo-free).
  void apply(const DevSell& Afine, const double* r, double* z);
  // The cycle in its own precision T (float for the mixed-precision cycle): right-hand side buffer of the
  // fine level (n rows) and one V-cycle on it; returns the solution vector.  Used for the replicated
  // coarse part of a distributed hierarchy.
  template <class T> T* rhs_buffer();
  template <class T> const T* cycle(const DevSell& Afine);
  bool fp32() const;
  // micro-benchmark hook: one smoothing step (SpMV fused with the Chebyshev recurrence) of level `level` on
  // the cycle's own vectors; rows / stored entries of that level's operator are returned for the roofline
  bool launch_level_smoother(int level, const DevSell& Afine, int64_t* rows, int64_t* nnz, int* value_bytes = nullptr);
  // the same for level `level`'s other SELL kernels, launched as the cycle launches them: which = 1 residual,
  // 2 restriction onto level + 1, 3 prolongation from level + 1 (0: the smoothing step).  info = {rows, columns,
  // stored entries, longest row, bytes per value of the matrix, bytes per vector entry, 1 if the restriction
  // also takes the coarse level's first Chebyshev step}.  false: no such kernel on this rank.
  bool launch_level_kernel(int level, int which, const DevSell& Afine, int64_t info[7]);
  // ---- test hooks (one rank; the shakti_amg_* functions of the C ABI).  false: no such level / matrix.
  // info: the layout of shakti_amg_level_info (shakti_b200.h)
  bool level_info(int level, const DevSell& Afine, int64_t info[18]) const;
  // matrix `which` of level `level` (0 A, 1 P, 2 R, 3 the fp32 copy of A, 4 the fp16 copy of D^-1 A) as a CSR in the
  // level's numbering, values widened to double
  bool level_matrix(int level, int which, const DevSell& Afine, HostCsr& csr, std::vector<double>& val) const;
  // the level's smoother diagonal in fp64 and in the cycle's precision, its Chebyshev bound and coefficients
  // (amg_cheby_coef_kernel: stride doubles; empty without the Chebyshev smoother)
  bool level_vectors(int level, std::vector<double>& dinv, std::vector<double>& dinv_cycle, double& lmax,
                     std::vector<double>& coef, int& stride) const;
  int levels() const;
  double operator_complexity() const;
  int64_t refreshes() const { return refreshes_; }
  bool ready() const { return refreshes_ > 0; }

 public:
  struct Impl;

 private:
  std::unique_ptr<Impl> p_;
  int64_t refreshes_ = 0;
};

}  // namespace shakti
