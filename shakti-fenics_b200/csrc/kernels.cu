// Hand-written sm_100a kernels of the SHAKTI hot path: transmissivity integral, residual +
// Jacobian assembly, nodal updates, SELL SpMV family and the vector kernels of the Krylov
// solvers.  All fp64 / int32, HBM-bandwidth bound by design (no tensor cores: nothing here is
// a dense contraction).  Reference formulas: source/constitutive.py:6-31, source/solvers.py:35-45.
#include <algorithm>
#include <cstdlib>
#include <ctime>

#include "device.h"

namespace shakti {

int64_t g_kernel_launches = 0;

bool pdl_enabled() {
  // on by default (measured at C4: -0.6 % of a step on one B200, -2.5 % on eight); SHAKTI_PDL=0 launches plainly
  static const bool on = getenv("SHAKTI_PDL") == nullptr || atoi(getenv("SHAKTI_PDL")) != 0;
  return on;
}

// ---- diagnostic phase timer (common.h)
static std::vector<std::pair<std::string, std::pair<double, int64_t>>> g_phases;
bool phase_trace_enabled() {
  static const bool on = getenv("SHAKTI_TRACE_PHASES") != nullptr;
  return on;
}
static double now_ms() {
  timespec ts;
  clock_gettime(CLOCK_MONOTONIC, &ts);
  return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6;
}
void phase_add(const char* name, double ms) {
  for (auto& p : g_phases)
    if (p.first == name) { p.second.first += ms; p.second.second++; return; }
  g_phases.push_back({name, {ms, 1}});
}
void phase_report(const char* title) {
  if (g_phases.empty()) return;
  fprintf(stderr, "[phases] %s:", title);
  for (auto& p : g_phases) fprintf(stderr, " %s=%.2fms/%lld", p.first.c_str(), p.second.first, (long long)p.second.second);
  fprintf(stderr, "\n");
  g_phases.clear();
}
PhaseScope::PhaseScope(const char* n, cudaStream_t st) : name(n), s(st), on(phase_trace_enabled()) {
  if (!on) return;
  cudaStreamSynchronize(s);
  t0 = now_ms();
}
PhaseScope::~PhaseScope() {
  if (!on) return;
  cudaStreamSynchronize(s);
  phase_add(name, now_ms() - t0);
}

DevParams make_dev_params(const shakti_params& p) {
  DevParams d;
  d.g = p.g; d.rho_i = p.rho_i; d.rho_w = p.rho_w; d.nu = p.nu; d.Lh = p.Lh;
  d.omega = p.omega; d.n = p.n; d.A = p.A;
  d.cm = 1.0 / p.rho_i - 1.0 / p.rho_w;
  d.rwg = p.rho_w * p.g;
  d.inv_rwg = 1.0 / d.rwg;
  d.inv_Lh = 1.0 / p.Lh;
  d.cm_over_Lh = d.cm / p.Lh;
  d.n_is_3 = (p.n == 3.0);
  return d;
}

void DevSell::upload_pattern(const HostSell& h, int64_t nnz_) {
  n_rows = (int32_t)h.n_rows; n_cols = (int32_t)h.n_cols; n_slices = (int32_t)h.n_slices;
  padded = h.padded(); nnz = nnz_;
  max_width = 0;
  for (int32_t l : h.rowlen) max_width = std::max(max_width, l);
  slice_ptr.upload(h.slice_ptr);
  col.upload(h.col);
  rowlen.upload(h.rowlen);
  val.alloc_zero(padded);
}

// ------------------------------------------------------------------ quadrature tables
constexpr int kMaxQ = 64;
__constant__ double c_kq[4 * kMaxQ];   // l0,l1,l2,w per point: rule for the K integral
__constant__ int c_nkq;
__constant__ double c_rq[4 * kMaxQ];   // rule for the closure/storage (reaction) integrals
__constant__ int c_nrq;

static void pack_rule(int n, const double* pts, const double* wts, double* out) {
  for (int k = 0; k < n; ++k) {
    out[4 * k + 0] = 1.0 - pts[2 * k] - pts[2 * k + 1];
    out[4 * k + 1] = pts[2 * k];
    out[4 * k + 2] = pts[2 * k + 1];
    out[4 * k + 3] = wts[k];
  }
}
void upload_k_rule(int n, const double* pts, const double* wts, cudaStream_t s) {
  SHAKTI_REQUIRE(n > 0 && n <= kMaxQ, "quadrature table must have 1..64 points");
  double h[4 * kMaxQ];
  pack_rule(n, pts, wts, h);
  SHAKTI_CUDA(cudaStreamSynchronize(s));
  SHAKTI_CUDA(cudaMemcpyToSymbol(c_kq, h, sizeof(double) * 4 * n));
  SHAKTI_CUDA(cudaMemcpyToSymbol(c_nkq, &n, sizeof(int)));
}
void upload_reaction_rule(int n, const double* pts, const double* wts, cudaStream_t s) {
  SHAKTI_REQUIRE(n > 0 && n <= kMaxQ, "quadrature table must have 1..64 points");
  double h[4 * kMaxQ];
  pack_rule(n, pts, wts, h);
  SHAKTI_CUDA(cudaStreamSynchronize(s));
  SHAKTI_CUDA(cudaMemcpyToSymbol(c_rq, h, sizeof(double) * 4 * n));
  SHAKTI_CUDA(cudaMemcpyToSymbol(c_nrq, &n, sizeof(int)));
}

// ------------------------------------------------------------------ element geometry
struct Geo {
  double gx[3], gy[3];  // grad phi_a
  double detabs;        // |det J| = 2 |T|
};

__device__ __forceinline__ Geo geometry(double x0, double y0, double x1, double y1, double x2, double y2) {
  Geo g;
  const double d1x = x1 - x0, d1y = y1 - y0, d2x = x2 - x0, d2y = y2 - y0;
  const double det = d1x * d2y - d2x * d1y;
  const double inv = 1.0 / det;
  g.gx[1] = d2y * inv;  g.gy[1] = -d2x * inv;
  g.gx[2] = -d1y * inv; g.gy[2] = d1x * inv;
  g.gx[0] = -g.gx[1] - g.gx[2];
  g.gy[0] = -g.gy[1] - g.gy[2];
  g.detabs = fabs(det);
  return g;
}

__device__ __forceinline__ double powabs(double a, double e, int e_is_2) {
  // |a|^e ; the n == 3 fast path keeps closure terms polynomial (abs(N)**(n-1), constitutive.py:31)
  return e_is_2 ? a * a : pow(fabs(a), e);
}

// ------------------------------------------------------------------ Kbar
// Kbar_T = |detJ| sum_k w_k K(b(xi_k), |q(xi_k)|),  K = |b|^3 g / (12 nu (1 + omega Re)),
// Re = sqrt(q.q)/nu   (constitutive.py:11-20).  One thread per cell; compute heavy
// (nq x (sqrt + div)) but executed once per time step because b, q are lagged (solvers.py:37-45).
__global__ void __launch_bounds__(256)
kbar_kernel(int32_t ne, const int32_t* __restrict__ c0, const int32_t* __restrict__ c1,
            const int32_t* __restrict__ c2, const double* __restrict__ x, const double* __restrict__ y,
            const double* __restrict__ b, const double* __restrict__ qx, const double* __restrict__ qy,
            double* __restrict__ kbar, DevParams p) {
  const int32_t e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= ne) return;
  const int32_t v0 = c0[e], v1 = c1[e], v2 = c2[e];
  const double x0 = x[v0], y0 = y[v0], x1 = x[v1], y1 = y[v1], x2 = x[v2], y2 = y[v2];
  const double detabs = fabs((x1 - x0) * (y2 - y0) - (x2 - x0) * (y1 - y0));
  const double b0 = b[v0], b1 = b[v1], b2 = b[v2];
  const double qx0 = qx[v0], qx1 = qx[v1], qx2 = qx[v2];
  const double qy0 = qy[v0], qy1 = qy[v1], qy2 = qy[v2];
  const double cK = p.g / (12.0 * p.nu);
  const double cRe = p.omega / p.nu;
  double acc = 0.0;
  const int nq = c_nkq;
  for (int k = 0; k < nq; ++k) {
    const double l0 = c_kq[4 * k], l1 = c_kq[4 * k + 1], l2 = c_kq[4 * k + 2], w = c_kq[4 * k + 3];
    const double bq = fabs(l0 * b0 + l1 * b1 + l2 * b2);
    const double u = l0 * qx0 + l1 * qx1 + l2 * qx2;
    const double v = l0 * qy0 + l1 * qy1 + l2 * qy2;
    const double qn = sqrt(u * u + v * v);
    acc += w * (bq * bq * bq) * cK / (1.0 + cRe * qn);
  }
  kbar[e] = acc * detabs;
}

void launch_kbar(int32_t ne, const int32_t* c0, const int32_t* c1, const int32_t* c2, const double* x,
                 const double* y, const double* b, const double* qx, const double* qy, double* kbar,
                 DevParams p, cudaStream_t s) {
  if (ne == 0) return;
  SHAKTI_LAUNCH(kbar_kernel, div_up(ne, 256), 256, 0, s, ne, c0, c1, c2, x, y, b, qx, qy, kbar, p);
}

// ------------------------------------------------------------------ element residual + Jacobian
// F_a  = Kbar (grad h . grad phi_a) + int [c_m Melt - Closure - storage/(rho_w g dt)(N-N_n) - inputs] phi_a
// J_ab = -Kbar/(rho_w g) grad phi_a.grad phi_b
//        + int [ c_m (q.grad phi_b)/Lh - (dClosure/dN + storage/(rho_w g dt)) phi_b ] phi_a
// (solvers.py:35-45,51).  grad h, grad b, grad melt are cell constants, so the Melt and inputs
// parts are P1 functions integrated in closed form (int phi_a phi_b = |detJ|/24 (1+delta_ab));
// closure (degree 5 for n = 3) and storage use the reaction rule in __constant__ memory.
struct ElemOut {
  double F[3];
  double J[3][3];
};

// closure (A b N^3, its N-derivative) and lake-storage terms of one cell by Radon's 7-point rule
// (see element_core); ST = false leaves the storage part out (cells with no storage).
template <bool ST>
__device__ __forceinline__ void reaction_radon7(double detabs, const double bb[3], const double Nv[3], const double Nn[3],
                                                const double st[3], double cs, double A, double& f0, double& f1, double& f2,
                                                double& m00, double& m01, double& m02, double& m11, double& m12, double& m22) {
  double dqv[3] = {0, 0, 0}, sv[3] = {0, 0, 0}, Sd = 0, Ss = 0;
  if (ST) {
#pragma unroll
    for (int i = 0; i < 3; ++i) { dqv[i] = Nv[i] - Nn[i]; sv[i] = st[i] * cs; }
    Sd = dqv[0] + dqv[1] + dqv[2];
    Ss = sv[0] + sv[1] + sv[2];
  }
  const double Sb = bb[0] + bb[1] + bb[2], SN = Nv[0] + Nv[1] + Nv[2];
  const double A3 = 3.0 * A;
  {  // centroid, weight 9/80
    const double w = 0.1125 * detabs, t = 1.0 / 3.0;
    const double bq = Sb * t, Nq = SN * t, N2 = Nq * Nq;
    double r = A * bq * Nq * N2, d = A3 * bq * N2;
    if (ST) {
      const double dq = Sd * t, sq = Ss * t;
      r += sq * dq;
      d += sq;
    }
    r *= w * t;
    d *= w * (t * t);
    f0 = f1 = f2 = r;
    m00 = m01 = m02 = m11 = m12 = m22 = d;
  }
  const double s15 = 3.872983346207417;   // sqrt(15)
#pragma unroll
  for (int orb = 0; orb < 2; ++orb) {
    const double a = orb == 0 ? (6.0 - s15) / 21.0 : (6.0 + s15) / 21.0;
    const double w = (orb == 0 ? (155.0 - s15) : (155.0 + s15)) * (1.0 / 2400.0) * detabs;
    const double e = 1.0 - 3.0 * a;   // c - a
    const double ab = a * Sb, aN = a * SN, ad = a * Sd, as = a * Ss;
    double r[3], d[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      const double bq = ab + e * bb[i], Nq = aN + e * Nv[i];
      const double N2 = Nq * Nq;
      double ri = A * bq * Nq * N2, di = A3 * bq * N2;
      if (ST) {
        const double dq = ad + e * dqv[i], sq = as + e * sv[i];
        ri += sq * dq;
        di += sq;
      }
      r[i] = w * ri;
      d[i] = w * di;
    }
    const double R = a * (r[0] + r[1] + r[2]), D = a * a * (d[0] + d[1] + d[2]);
    const double ae = a * e, ee = e * e;
    f0 += R + e * r[0]; f1 += R + e * r[1]; f2 += R + e * r[2];
    m00 += D + (2.0 * ae + ee) * d[0];
    m11 += D + (2.0 * ae + ee) * d[1];
    m22 += D + (2.0 * ae + ee) * d[2];
    m01 += D + ae * (d[0] + d[1]);
    m02 += D + ae * (d[0] + d[2]);
    m12 += D + ae * (d[1] + d[2]);
  }
}

__device__ __forceinline__ void element_core(const Geo& g, const double h[3], const double bb[3], const double mm[3],
                                             const double qxv[3], const double qyv[3], const double Nv[3],
                                             const double Nn[3], const double st[3], const double Gv[3],
                                             const double inp[3], double kb, double dt, const DevParams& p, ElemOut& o) {
  double ghx = 0, ghy = 0, gbx = 0, gby = 0, gmx = 0, gmy = 0;
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    ghx += h[i] * g.gx[i];  ghy += h[i] * g.gy[i];
    gbx += bb[i] * g.gx[i]; gby += bb[i] * g.gy[i];
    gmx += mm[i] * g.gx[i]; gmy += mm[i] * g.gy[i];
  }
  const double gb2 = gbx * gbx + gby * gby;
  const double gmgb = gmx * gbx + gmy * gby;
  const double inv1 = 1.0 / (1.0 + gb2);
  // nodal values of the P1 part of the reaction integrand
  double rl[3], rsum = 0, qxs = 0, qys = 0;
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const double m0 = (Gv[i] - p.rwg * (qxv[i] * ghx + qyv[i] * ghy)) * p.inv_Lh;   // constitutive.py:25
    const double md = (gb2 * mm[i] + bb[i] * gmgb) * inv1;                           // constitutive.py:26
    rl[i] = p.cm * (m0 + md) - inp[i];
    rsum += rl[i];
    qxs += qxv[i];
    qys += qyv[i];
  }
  const double m24 = g.detabs * (1.0 / 24.0);
  const double kJ = -kb * p.inv_rwg;
  const double cadv = p.cm_over_Lh * m24;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    o.F[a] = kb * (ghx * g.gx[a] + ghy * g.gy[a]) + m24 * (rsum + rl[a]);
    const double qax = cadv * (qxs + qxv[a]), qay = cadv * (qys + qyv[a]);
#pragma unroll
    for (int b = 0; b < 3; ++b)
      o.J[a][b] = kJ * (g.gx[a] * g.gx[b] + g.gy[a] * g.gy[b]) + qax * g.gx[b] + qay * g.gy[b];
  }
  // closure + storage by quadrature
  const double cs = p.inv_rwg / dt;
  double f0 = 0, f1 = 0, f2 = 0, m00 = 0, m01 = 0, m02 = 0, m11 = 0, m12 = 0, m22 = 0;
  if (p.n_is_3) {
    // n = 3: integrands are polynomials of degree <= 5 -> Radon's 7-point rule, written out by orbit.
    // A P1 function with nodal values f_i and sum S is  S/3 at the centroid and  a S + (c-a) f_i  at
    // orbit point i (barycentrics (a,a,c) permuted), so every interpolation is one FMA; the
    // phi_a, phi_a phi_b weights collapse to  a R + e r_a  and  a^2 D + a e (d_a + d_b) + e^2 delta_ab d_a.
    // Cells outside the lakes (storage == 0 at all three vertices: almost all of them) skip the storage
    // interpolations; the branch is uniform over long runs of cells.
    if (st[0] != 0.0 || st[1] != 0.0 || st[2] != 0.0)
      reaction_radon7<true>(g.detabs, bb, Nv, Nn, st, cs, p.A, f0, f1, f2, m00, m01, m02, m11, m12, m22);
    else
      reaction_radon7<false>(g.detabs, bb, Nv, Nn, st, cs, p.A, f0, f1, f2, m00, m01, m02, m11, m12, m22);
  } else {
    // general Glen exponent: the closure is not polynomial; use the table in __constant__ memory
    const double e1 = p.n - 1.0, e2 = p.n - 2.0;
    const int nq = c_nrq;
    for (int k = 0; k < nq; ++k) {
      const double l0 = c_rq[4 * k], l1 = c_rq[4 * k + 1], l2 = c_rq[4 * k + 2];
      const double w = c_rq[4 * k + 3] * g.detabs;
      const double bq = l0 * bb[0] + l1 * bb[1] + l2 * bb[2];
      const double Nq = l0 * Nv[0] + l1 * Nv[1] + l2 * Nv[2];
      const double dq = Nq - (l0 * Nn[0] + l1 * Nn[1] + l2 * Nn[2]);
      const double sq = (l0 * st[0] + l1 * st[1] + l2 * st[2]) * cs;
      const double sgn = Nq > 0 ? 1.0 : (Nq < 0 ? -1.0 : 0.0);
      const double p1 = pow(fabs(Nq), e1);
      const double clos = p.A * bq * Nq * p1;
      const double dclos = p.A * bq * (p1 + Nq * e1 * pow(fabs(Nq), e2) * sgn);
      const double r = w * (clos + sq * dq);
      const double d = w * (dclos + sq);
      f0 += r * l0; f1 += r * l1; f2 += r * l2;
      const double d0 = d * l0, d1 = d * l1;
      m00 += d0 * l0; m01 += d0 * l1; m02 += d0 * l2;
      m11 += d1 * l1; m12 += d1 * l2; m22 += d * l2 * l2;
    }
  }
  o.F[0] -= f0; o.F[1] -= f1; o.F[2] -= f2;
  o.J[0][0] -= m00; o.J[0][1] -= m01; o.J[0][2] -= m02;
  o.J[1][0] -= m01; o.J[1][1] -= m11; o.J[1][2] -= m12;
  o.J[2][0] -= m02; o.J[2][1] -= m12; o.J[2][2] -= m22;
}

// vertex data gathered straight from global memory (cell-parallel variant)
__device__ __forceinline__ void element_FJ(const int32_t v[3], const FieldPtrs& f, double kb, double dt,
                                           const DevParams& p, ElemOut& o, double Nv[3]) {
  const Geo g = geometry(f.x[v[0]], f.y[v[0]], f.x[v[1]], f.y[v[1]], f.x[v[2]], f.y[v[2]]);
  double h[3], bb[3], mm[3], qxv[3], qyv[3], Nn[3], st[3], Gv[3], inp[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    Nv[i] = f.N[v[i]];
    h[i] = f.h0[v[i]] - Nv[i] * p.inv_rwg;
    bb[i] = f.b[v[i]];
    mm[i] = f.melt[v[i]];
    qxv[i] = f.qx[v[i]];
    qyv[i] = f.qy[v[i]];
    Nn[i] = f.N_n[v[i]];
    st[i] = f.storage[v[i]];
    Gv[i] = f.G[v[i]];
    inp[i] = f.inputs[v[i]];
  }
  element_core(g, h, bb, mm, qxv, qyv, Nv, Nn, st, Gv, inp, kb, dt, p, o);
}

// Dirichlet lifting (scale -1: F += J_full (g - x) on bc columns) applied in place.
__device__ __forceinline__ void apply_lifting(ElemOut& o, const double Nv[3], const bool bc[3], double N_bdry) {
#pragma unroll
  for (int b = 0; b < 3; ++b)
    if (bc[b]) {
      const double gx = N_bdry - Nv[b];
#pragma unroll
      for (int a = 0; a < 3; ++a) o.F[a] += o.J[a][b] * gx;
    }
}

// Same element computation with the vertex data already staged in shared memory
// (sV[field][vcap], field order of enum VX..VI below; VH holds the head h, not h0).
__device__ __forceinline__ void element_FJ_staged(const int v[3], const double* __restrict__ sV, int vcap, double kb,
                                                  double dt, const DevParams& p, ElemOut& o, double Nv[3]) {
  const Geo g = geometry(sV[0 * vcap + v[0]], sV[1 * vcap + v[0]], sV[0 * vcap + v[1]], sV[1 * vcap + v[1]],
                         sV[0 * vcap + v[2]], sV[1 * vcap + v[2]]);
  double h[3], bb[3], mm[3], qxv[3], qyv[3], Nn[3], st[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    h[i] = sV[2 * vcap + v[i]];
    Nv[i] = sV[3 * vcap + v[i]];
    Nn[i] = sV[4 * vcap + v[i]];
    bb[i] = sV[5 * vcap + v[i]];
    qxv[i] = sV[6 * vcap + v[i]];
    qyv[i] = sV[7 * vcap + v[i]];
    mm[i] = sV[9 * vcap + v[i]];
    st[i] = sV[10 * vcap + v[i]];
  }
  double Gv[3], inp[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) { Gv[i] = sV[8 * vcap + v[i]]; inp[i] = sV[11 * vcap + v[i]]; }
  element_core(g, h, bb, mm, qxv, qyv, Nv, Nn, st, Gv, inp, kb, dt, p, o);
}

// Variant 1: one thread per cell, scatter with fp64 atomics into the SELL value array through
// the precomputed (cell, a, b) -> position table.  F and Jval must be zeroed beforehand.
__global__ void __launch_bounds__(128)
assemble_atomic_kernel(int32_t ne, int32_t n_owned, const int32_t* __restrict__ c0,
                       const int32_t* __restrict__ c1, const int32_t* __restrict__ c2,
                       const int32_t* __restrict__ slot, FieldPtrs f, const double* __restrict__ kbar,
                       double dt, double N_bdry, double* __restrict__ F, double* __restrict__ Jval,
                       int want_J, DevParams p) {
  const int32_t e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= ne) return;
  const int32_t v[3] = {c0[e], c1[e], c2[e]};
  ElemOut o;
  double Nv[3];
  element_FJ(v, f, kbar[e], dt, p, o, Nv);
  const bool bc[3] = {f.isbc[v[0]] != 0, f.isbc[v[1]] != 0, f.isbc[v[2]] != 0};
  apply_lifting(o, Nv, bc, N_bdry);
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    if (v[a] >= n_owned || bc[a]) continue;   // owner computes; bc rows are set by apply_bc
    atomicAdd(&F[v[a]], o.F[a]);
    if (want_J) {
#pragma unroll
      for (int b = 0; b < 3; ++b)
        if (!bc[b]) atomicAdd(&Jval[slot[(size_t)(3 * a + b) * ne + e]], o.J[a][b]);
    }
  }
}

void launch_assemble_atomic(int32_t ne, int32_t n_owned, const int32_t* c0, const int32_t* c1,
                            const int32_t* c2, const int32_t* slot, FieldPtrs f, const double* kbar,
                            double dt, double N_bdry, double* F, double* Jval, int want_J, DevParams p,
                            cudaStream_t s) {
  if (ne == 0) return;
  SHAKTI_LAUNCH(assemble_atomic_kernel, div_up(ne, 128), 128, 0, s, ne, n_owned, c0, c1, c2, slot, f, kbar,
                dt, N_bdry, F, Jval, want_J, p);
}

// Variant 0 (default): atomics-free row-block assembly.  A CUDA block owns a run of consecutive
// rows (= whole SELL slices).
//   Phase 0: the twelve vertex fields of the block's vertices (its own rows: contiguous, fully
//            coalesced; plus the few halo vertices of its cells) are staged in shared memory.
//   Phase 1: every cell touching those rows is computed from shared memory and its 3 + 9
//            numbers are staged in shared memory (structure of arrays, conflict free).  Cells on
//            block borders are computed by each block that needs them (~19 % extra at 256 rows).
//   Phase 2: one thread per row gathers -- the residual and the diagonal from the row's incident
//            cells, every off-diagonal entry from the (at most two) cells sharing that edge -- and
//            writes the SELL values with plain coalesced stores.
// No zero-fill, no atomics, bitwise reproducible.
enum { VX = 0, VY, VH, VN, VNN, VB, VQX, VQY, VG, VM, VS, VI, VFIELDS };

__global__ void __launch_bounds__(256, 2)
assemble_blocks_kernel(int32_t n_owned, int32_t rows_per_block, int32_t cap, int32_t vcap,
                       const int32_t* __restrict__ blk_eptr, const int32_t* __restrict__ blk_elems,
                       const uint16_t* __restrict__ blk_lv, const int32_t* __restrict__ blk_hptr,
                       const int32_t* __restrict__ blk_halo, const int32_t* __restrict__ inc_ptr,
                       const uint16_t* __restrict__ inc_code, const uint32_t* __restrict__ src, FieldPtrs f,
                       const double* __restrict__ kbar, double dt, double N_bdry, const int32_t* __restrict__ slice_ptr,
                       double* __restrict__ F, double* __restrict__ Jval, int want_J, DevParams p) {
  extern __shared__ double smem[];
  double* sV = smem;                         // [VFIELDS][vcap]
  double* sK = smem + (size_t)VFIELDS * vcap;  // [12][cap]: F0..F2, J00..J22
  uint8_t* sBC = reinterpret_cast<uint8_t*>(sK + (size_t)12 * cap);   // [vcap]
  const int32_t r0 = blockIdx.x * rows_per_block;
  const int32_t nrows = min(rows_per_block, n_owned - r0);
  const int32_t h0 = blk_hptr[blockIdx.x], nh = blk_hptr[blockIdx.x + 1] - h0;
  // cell ids, Kbar and block-local vertex ids of this thread's cells are requested first: the chain
  // blk_elems -> kbar would otherwise be exposed at the start of every cell (low occupancy)
  constexpr int kCellsPre = 4;
  const int32_t e0 = blk_eptr[blockIdx.x], e1 = blk_eptr[blockIdx.x + 1];
  double kb_pre[kCellsPre];
  uint32_t lv01_pre[kCellsPre], lv2_pre[kCellsPre];
#pragma unroll
  for (int c = 0; c < kCellsPre; ++c) {
    const int32_t le = threadIdx.x + c * blockDim.x;
    kb_pre[c] = 0.0; lv01_pre[c] = 0; lv2_pre[c] = 0;
    if (le < e1 - e0) {
      const uint16_t* lv = blk_lv + 3 * (size_t)(e0 + le);
      lv01_pre[c] = (uint32_t)lv[0] | ((uint32_t)lv[1] << 16);
      lv2_pre[c] = lv[2];
      kb_pre[c] = kbar[blk_elems[e0 + le]];
    }
  }
  // ---- phase 0
  for (int32_t i = threadIdx.x; i < nrows + nh; i += blockDim.x) {
    const int32_t g = i < nrows ? r0 + i : blk_halo[h0 + i - nrows];
    const double Ni = f.N[g];
    sV[VX * vcap + i] = f.x[g];
    sV[VY * vcap + i] = f.y[g];
    sV[VH * vcap + i] = f.h0[g] - Ni * p.inv_rwg;   // Head (constitutive.py:6-9)
    sV[VN * vcap + i] = Ni;
    sV[VNN * vcap + i] = f.N_n[g];
    sV[VB * vcap + i] = f.b[g];
    sV[VQX * vcap + i] = f.qx[g];
    sV[VQY * vcap + i] = f.qy[g];
    sV[VG * vcap + i] = f.G[g];
    sV[VM * vcap + i] = f.melt[g];
    sV[VS * vcap + i] = f.storage[g];
    sV[VI * vcap + i] = f.inputs[g];
    sBC[i] = f.isbc[g];
  }
  __syncthreads();
  // ---- phase 1
#pragma unroll 1
  for (int c = 0; c * (int32_t)blockDim.x + (int32_t)threadIdx.x < e1 - e0; ++c) {
    const int32_t le = threadIdx.x + c * blockDim.x;
    int v[3];
    double kb;
    if (c < kCellsPre) {
      uint32_t a01 = lv01_pre[0], a2 = lv2_pre[0];
      kb = kb_pre[0];
#pragma unroll
      for (int q = 1; q < kCellsPre; ++q)
        if (c == q) { a01 = lv01_pre[q]; a2 = lv2_pre[q]; kb = kb_pre[q]; }
      v[0] = a01 & 0xFFFFu; v[1] = a01 >> 16; v[2] = a2;
    } else {
      const uint16_t* lv = blk_lv + 3 * (size_t)(e0 + le);
      v[0] = lv[0]; v[1] = lv[1]; v[2] = lv[2];
      kb = kbar[blk_elems[e0 + le]];
    }
    ElemOut o;
    double Nv[3];
    element_FJ_staged(v, sV, vcap, kb, dt, p, o, Nv);
    const bool bc[3] = {sBC[v[0]] != 0, sBC[v[1]] != 0, sBC[v[2]] != 0};
    apply_lifting(o, Nv, bc, N_bdry);
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      sK[a * cap + le] = o.F[a];
#pragma unroll
      for (int b = 0; b < 3; ++b) sK[(3 + 3 * a + b) * cap + le] = (bc[a] || bc[b]) ? 0.0 : o.J[a][b];
    }
  }
  // ---- phase 2 (its first loads are issued before the barrier so that they are in flight while
  // the block's last cells finish: the gather codes of the row's first kPre entries and the bounds
  // of its incident-cell list)
  constexpr int kPre = 8;
  const bool has_row = (int32_t)threadIdx.x < nrows;
  const int32_t row = r0 + threadIdx.x;
  int32_t base = 0, w = 0, ib = 0, ie = 0;
  uint32_t pre[kPre];
  if (has_row) {
    const int32_t slice = row >> 5;
    base = slice_ptr[slice];
    w = (slice_ptr[slice + 1] - base) >> 5;
    ib = inc_ptr[row];
    ie = inc_ptr[row + 1];
    if (want_J) {
#pragma unroll
      for (int k = 0; k < kPre; ++k) pre[k] = k < w ? src[base + 32 * k + (row & 31)] : 0xFFFFFFFFu;
    }
  }
  __syncthreads();
  if (!has_row) return;
  const bool rbc = sBC[threadIdx.x] != 0;
  double Fr = 0.0, Jd = 0.0;
  for (int32_t k = ib; k < ie; ++k) {
    const uint32_t code = inc_code[k];
    const uint32_t le = code >> 2, a = code & 3u;
    Fr += sK[a * cap + le];
    Jd += sK[(3 + 4 * a) * cap + le];
  }
  F[row] = rbc ? sV[VN * vcap + threadIdx.x] - N_bdry : Fr;
  if (!want_J) return;
  auto entry = [&](uint32_t s2, int32_t pos) {
    if (s2 == 0xFFFFFFFFu) return;         // padding
    double v;
    if (s2 == 0xFFFEFFFEu) v = rbc ? 1.0 : Jd;
    else {
      const uint32_t ca = s2 & 0xFFFFu, cb = s2 >> 16;
      v = sK[(3 + (ca & 15u)) * cap + (ca >> 4)];
      if (cb != 0xFFFFu) v += sK[(3 + (cb & 15u)) * cap + (cb >> 4)];
    }
    Jval[pos] = v;
  };
#pragma unroll
  for (int k = 0; k < kPre; ++k)
    if (k < w) entry(pre[k], base + 32 * k + (row & 31));
  for (int k = kPre; k < w; ++k) {
    const int32_t pos = base + 32 * k + (row & 31);
    entry(src[pos], pos);
  }
}

void launch_assemble_blocks(const AssemblyPlanView& pl, FieldPtrs f, const double* kbar, double dt, double N_bdry,
                            const int32_t* slice_ptr, double* F, double* Jval, int want_J, DevParams p, cudaStream_t s) {
  if (pl.n_blocks == 0) return;
  int dev = 0;
  SHAKTI_CUDA(cudaGetDevice(&dev));
  const size_t smem = ((size_t)VFIELDS * pl.vcap + (size_t)12 * pl.cap) * sizeof(double) + pl.vcap;
  static size_t configured[64] = {};    // per device (a process may drive several GPUs)
  if (smem > configured[dev & 63]) {
    SHAKTI_CUDA(cudaFuncSetAttribute(assemble_blocks_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured[dev & 63] = smem;
  }
  const int threads = pl.rows_per_block >= 256 ? 256 : 128;   // phase 2 needs one thread per row
  SHAKTI_LAUNCH(assemble_blocks_kernel, pl.n_blocks, threads, smem, s, pl.n_owned, pl.rows_per_block, pl.cap, pl.vcap,
                pl.blk_eptr, pl.blk_elems, pl.blk_lv, pl.blk_hptr, pl.blk_halo, pl.inc_ptr, pl.inc_code, pl.src, f, kbar, dt,
                N_bdry, slice_ptr, F, Jval, want_J, p);
}

// F[bc] = N[bc] - g ; J[bc,bc] = 1  (DOLFINx set_bc with scale -1 / insert_diagonal)
__global__ void apply_bc_kernel(int32_t n_owned, const uint8_t* __restrict__ isbc, const double* __restrict__ N,
                                double N_bdry, const int32_t* __restrict__ diag_pos, double* __restrict__ F,
                                double* __restrict__ Jval, int want_J) {
  const int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_owned || !isbc[i]) return;
  F[i] = N[i] - N_bdry;
  if (want_J) Jval[diag_pos[i]] = 1.0;
}
void launch_apply_bc(int32_t n_owned, const uint8_t* isbc, const double* N, double N_bdry,
                     const int32_t* diag_pos, double* F, double* Jval, int want_J, cudaStream_t s) {
  if (n_owned == 0) return;
  SHAKTI_LAUNCH(apply_bc_kernel, div_up(n_owned, 256), 256, 0, s, n_owned, isbc, N, N_bdry, diag_pos, F, Jval, want_J);
}

// ------------------------------------------------------------------ nodal updates
// Function.interpolate(Expression): the value at vertex i comes from the highest-index cell
// containing i, evaluated with that cell's constant gradients (SURVEY.md rows a12-a14).
struct WinGeo {
  int32_t v[3];
  int loc;
  Geo g;
};
__device__ __forceinline__ WinGeo win_geometry(const int32_t* __restrict__ win, int32_t i,
                                               const double* __restrict__ x, const double* __restrict__ y) {
  WinGeo w;
  const int4 t = reinterpret_cast<const int4*>(win)[i];
  w.v[0] = t.x; w.v[1] = t.y; w.v[2] = t.z; w.loc = t.w;
  if (w.loc >= 0) w.g = geometry(x[t.x], y[t.x], x[t.y], y[t.y], x[t.z], y[t.z]);
  return w;
}
__device__ __forceinline__ void cell_grad(const WinGeo& w, const double f[3], double& gx, double& gy) {
  gx = f[0] * w.g.gx[0] + f[1] * w.g.gx[1] + f[2] * w.g.gx[2];
  gy = f[0] * w.g.gy[0] + f[1] * w.g.gy[1] + f[2] * w.g.gy[2];
}

__device__ __forceinline__ double melt_at_vertex(const WinGeo& w, int32_t i, const double* __restrict__ h0,
                                                 const double* __restrict__ N, const double* __restrict__ b,
                                                 const double* __restrict__ qx, const double* __restrict__ qy,
                                                 const double* __restrict__ G, const double* __restrict__ melt,
                                                 const DevParams& p) {
  double h[3], bb[3], mm[3];
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    h[a] = h0[w.v[a]] - N[w.v[a]] / p.rwg;
    bb[a] = b[w.v[a]];
    mm[a] = melt[w.v[a]];
  }
  double ghx, ghy, gbx, gby, gmx, gmy;
  cell_grad(w, h, ghx, ghy);
  cell_grad(w, bb, gbx, gby);
  cell_grad(w, mm, gmx, gmy);
  const double gb2 = gbx * gbx + gby * gby;
  const double m0 = (G[i] - p.rwg * (qx[i] * ghx + qy[i] * ghy)) / p.Lh;
  const double md = (gb2 * melt[i] + b[i] * (gmx * gbx + gmy * gby)) / (1.0 + gb2);
  return m0 + md;
}

// b <- max(b + dt (Melt(q_new, N_new, b_old, melt_new)/rho_i - A b N |N|^(n-1)), b_min)
// (solvers.py:162,192,196)
__global__ void __launch_bounds__(256)
update_b_kernel(int32_t n_owned, const int32_t* __restrict__ win, const double* __restrict__ x,
                const double* __restrict__ y, const double* __restrict__ h0, const double* __restrict__ N,
                const double* __restrict__ b_old, const double* __restrict__ qx, const double* __restrict__ qy,
                const double* __restrict__ G, const double* __restrict__ melt, double* __restrict__ b_new,
                double dt, double b_min, DevParams p) {
  const int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_owned) return;
  const WinGeo w = win_geometry(win, i, x, y);
  double bn;
  if (w.loc < 0) bn = b_old[i];
  else {
    const double m = melt_at_vertex(w, i, h0, N, b_old, qx, qy, G, melt, p);
    const double Ni = N[i];
    const double clos = p.A * b_old[i] * Ni * powabs(Ni, p.n - 1.0, p.n_is_3);
    bn = b_old[i] + dt * (m / p.rho_i - clos);
  }
  b_new[i] = bn < b_min ? b_min : bn;
}
void launch_update_b(int32_t n_owned, const int32_t* win, const double* x, const double* y, const double* h0,
                     const double* N, const double* b_old, const double* qx, const double* qy, const double* G,
                     const double* melt, double* b_new, double dt, double b_min, DevParams p, cudaStream_t s) {
  if (n_owned == 0) return;
  SHAKTI_LAUNCH(update_b_kernel, div_up(n_owned, 256), 256, 0, s, n_owned, win, x, y, h0, N, b_old, qx, qy, G,
                melt, b_new, dt, b_min, p);
}

// Pass 1 of the nodal updates (solvers.py:186,189):
//   q      <- -|b|^3 g grad h / (12 nu (1 + omega |q_old|/nu))        (solvers.py:143)
//   melt_n <- Melt(q_new, Head(N_new), G, b_old, melt_old)             (solvers.py:165)
// Q / MELT select the outputs; with Q false, q is read from memory.  The melt update at vertex i needs the NEW
// flux at i only, so with both on they come from one load of the winning cell, one geometry and one head
// gradient.  (The gap-height update needs the new melt at the cell's other vertices and therefore stays a
// second pass.)
template <bool Q, bool MELT>
__global__ void __launch_bounds__(256)
update_q_melt_kernel(int32_t n_owned, const int32_t* __restrict__ win, const double* __restrict__ x,
                     const double* __restrict__ y, const double* __restrict__ h0, const double* __restrict__ N,
                     const double* __restrict__ b, double* __restrict__ qx, double* __restrict__ qy,
                     const double* __restrict__ G, const double* __restrict__ melt_old, double* __restrict__ melt_new,
                     DevParams p) {
  const int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_owned) return;
  const WinGeo w = win_geometry(win, i, x, y);
  if (w.loc < 0) {
    if (MELT) melt_new[i] = melt_old[i];
    return;
  }
  double h[3], bb[3], mm[3] = {0.0, 0.0, 0.0};
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    h[a] = h0[w.v[a]] - N[w.v[a]] / p.rwg;
    bb[a] = b[w.v[a]];
    if (MELT) mm[a] = melt_old[w.v[a]];
  }
  double ghx, ghy, gbx, gby, gmx, gmy;
  cell_grad(w, h, ghx, ghy);
  cell_grad(w, bb, gbx, gby);
  cell_grad(w, mm, gmx, gmy);
  // the vertex's own values are those of its slot in the winning cell
  const double b_i = w.loc == 0 ? bb[0] : (w.loc == 1 ? bb[1] : bb[2]);
  const double m_i = w.loc == 0 ? mm[0] : (w.loc == 1 ? mm[1] : mm[2]);
  double qxn = qx[i], qyn = qy[i];
  if (Q) {
    const double bi = fabs(b_i);
    const double Re = sqrt(qxn * qxn + qyn * qyn) / p.nu;
    const double p1 = -(bi * bi * bi) * p.g;
    const double p2 = 12.0 * p.nu * (1.0 + p.omega * Re);
    qxn = p1 * ghx / p2;
    qyn = p1 * ghy / p2;
    qx[i] = qxn;
    qy[i] = qyn;
  }
  if (!MELT) return;
  const double gb2 = gbx * gbx + gby * gby;
  const double m0 = (G[i] - p.rwg * (qxn * ghx + qyn * ghy)) / p.Lh;
  const double md = (gb2 * m_i + b_i * (gmx * gbx + gmy * gby)) / (1.0 + gb2);
  melt_new[i] = m0 + md;
}
void launch_update_q(int32_t n_owned, const int32_t* win, const double* x, const double* y, const double* h0,
                     const double* N, const double* b, double* qx, double* qy, DevParams p, cudaStream_t s) {
  if (n_owned == 0) return;
  SHAKTI_LAUNCH((update_q_melt_kernel<true, false>), div_up(n_owned, 256), 256, 0, s, n_owned, win, x, y, h0, N, b, qx, qy,
                nullptr, nullptr, nullptr, p);
}
void launch_update_melt(int32_t n_owned, const int32_t* win, const double* x, const double* y, const double* h0,
                        const double* N, const double* b, const double* qx, const double* qy, const double* G,
                        const double* melt_old, double* melt_new, DevParams p, cudaStream_t s) {
  if (n_owned == 0) return;
  // with Q false the kernel only reads qx, qy
  SHAKTI_LAUNCH((update_q_melt_kernel<false, true>), div_up(n_owned, 256), 256, 0, s, n_owned, win, x, y, h0, N, b,
                const_cast<double*>(qx), const_cast<double*>(qy), G, melt_old, melt_new, p);
}
void launch_update_q_melt(int32_t n_owned, const int32_t* win, const double* x, const double* y, const double* h0,
                          const double* N, const double* b, double* qx, double* qy, const double* G,
                          const double* melt_old, double* melt_new, DevParams p, cudaStream_t s) {
  if (n_owned == 0) return;
  SHAKTI_LAUNCH((update_q_melt_kernel<true, true>), div_up(n_owned, 256), 256, 0, s, n_owned, win, x, y, h0, N, b, qx, qy,
                G, melt_old, melt_new, p);
}

// ------------------------------------------------------------------ SELL-32 SpMV family
// One thread per row, one warp per slice: entry k of the 32 rows of a slice is contiguous, so
// value/column loads are perfectly coalesced; x is gathered through L1/L2 (rows are Morton
// ordered, neighbours are close in memory).
enum { SPMV_SET = 0, SPMV_ADD = 1, SPMV_RESID = 2, SPMV_JACOBI = 3 };

// KG = 1: one thread per row (large matrices: enough rows to fill the GPU, loads of a warp coalesce over
// the 32 rows of a slice).  KG = 8: one 256-thread block per slice, warp g takes the entries k = g, g+8, ...
// of all 32 rows (still coalesced) and the eight partial sums meet in shared memory.  That is for the small,
// wide-rowed coarse levels of the AMG hierarchy, where one thread per row is a chain of ~100 dependent
// gathers (15 us for a 500-row level) and the eight-way split cuts the chain eightfold.  RB: row bound of the
// KG = 1 row product (sell_row.h), which amg.cu's one-thread-per-row kernels share.
template <class T, int KG, int RB>
__device__ __forceinline__ bool sell_row_dot(const SellViewT<T>& A, const T* __restrict__ x, int32_t& row, T& acc) {
  if (KG == 1) {
    row = blockIdx.x * blockDim.x + threadIdx.x;
    const int32_t slice = row >> 5;
    if (slice >= A.n_slices) return false;
    const int32_t base = A.slice_ptr[slice];
    const int32_t w = (A.slice_ptr[slice + 1] - base) >> 5;
    acc = sell_row_product<RB>(A.col + base + (row & 31), A.val + base + (row & 31), w, x);
    return row < A.n_rows;
  } else {
    __shared__ T psum[KG][32];
    const int32_t slice = blockIdx.x;
    const int lane = threadIdx.x & 31, g = threadIdx.x >> 5;
    row = slice * 32 + lane;
    const int32_t base = A.slice_ptr[slice];
    const int32_t w = (A.slice_ptr[slice + 1] - base) >> 5;
    const int32_t* __restrict__ cp = A.col + base + lane;
    const T* __restrict__ vp = A.val + base + lane;
    T a = 0;
    for (int k = g; k < w; k += KG) a += vp[32 * k] * x[cp[32 * k]];
    psum[g][lane] = a;
    __syncthreads();
    if (g != 0) return false;
#pragma unroll
    for (int j = 1; j < KG; ++j) a += psum[j][lane];
    acc = a;
    return row < A.n_rows;
  }
}
constexpr int32_t kWideRowsBelow = 300000;   // matrices with fewer rows use the KG = 8 kernels

template <int MODE, class T, int KG, int RB = 0>
__global__ void __launch_bounds__(256)
spmv_sell_kernel(SellViewT<T> A, const T* __restrict__ x, const T* __restrict__ b, const T* __restrict__ dinv, T omega,
                 T* __restrict__ y) {
  pdl_sync();
  int32_t row;
  T acc;
  if (!sell_row_dot<T, KG, RB>(A, x, row, acc)) return;
  if (MODE == SPMV_SET) y[row] = acc;
  else if (MODE == SPMV_ADD) y[row] += acc;
  else if (MODE == SPMV_RESID) y[row] = b[row] - acc;
  else y[row] = x[row] + omega * dinv[row] * (b[row] - acc);
}

template <int MODE, class T>
static void spmv_launch(SellViewT<T> A, const T* x, const T* b, const T* dinv, double omega, T* y, cudaStream_t s) {
  if (A.n_rows == 0) return;
  if (A.n_rows < kWideRowsBelow) {
    SHAKTI_LAUNCH_PDL((spmv_sell_kernel<MODE, T, 8>), A.n_slices, 256, 0, s, A, x, b, dinv, (T)omega, y);
    return;
  }
  sell_row_bound_dispatch<T>(A.max_width, [&](auto rb) {
    SHAKTI_LAUNCH_PDL((spmv_sell_kernel<MODE, T, 1, rb.value>), div_up((int64_t)A.n_slices * 32, 256), 256, 0, s, A, x, b, dinv, (T)omega, y);
  });
}
// Restriction that also takes the coarse level's first Chebyshev step from a zero guess: b_c = R r and
// x_c = (dinv_c b_c)/theta_c -- spmv_sell_kernel<SPMV_SET> and amg_cheby_first_kernel (amg.cu) in one pass,
// same operations in the same order.  d is not written; the coarse level's next sweep reads x_c in its place.
template <class T, int KG, int RB = 0>
__global__ void __launch_bounds__(256)
restrict_cheby_first_kernel(SellViewT<T> R, const T* __restrict__ r, const T* __restrict__ dinv_c,
                            const double* __restrict__ inv_theta, T* __restrict__ b_c, T* __restrict__ x_c) {
  pdl_sync();
  int32_t row;
  T acc;
  if (!sell_row_dot<T, KG, RB>(R, r, row, acc)) return;
  b_c[row] = acc;
  x_c[row] = dinv_c[row] * acc * (T)inv_theta[0];
}
template <class T>
void launch_restrict_cheby_first(SellViewT<T> R, const T* r, const T* dinv_c, const double* inv_theta, T* b_c, T* x_c, cudaStream_t s) {
  if (R.n_rows == 0) return;
  if (R.n_rows < kWideRowsBelow)
    SHAKTI_LAUNCH_PDL((restrict_cheby_first_kernel<T, 8>), R.n_slices, 256, 0, s, R, r, dinv_c, inv_theta, b_c, x_c);
  else
    sell_row_bound_dispatch<T>(R.max_width, [&](auto rb) {
      SHAKTI_LAUNCH_PDL((restrict_cheby_first_kernel<T, 1, rb.value>), div_up((int64_t)R.n_slices * 32, 256), 256, 0, s, R, r, dinv_c,
                        inv_theta, b_c, x_c);
    });
}
template void launch_restrict_cheby_first<double>(SellViewT<double>, const double*, const double*, const double*, double*, double*,
                                                  cudaStream_t);
template void launch_restrict_cheby_first<float>(SellViewT<float>, const float*, const float*, const double*, float*, float*,
                                                 cudaStream_t);

template <class T> void launch_spmv(SellViewT<T> A, const T* x, T* y, cudaStream_t s) { spmv_launch<SPMV_SET, T>(A, x, nullptr, nullptr, 0, y, s); }
template <class T> void launch_spmv_add(SellViewT<T> A, const T* x, T* y, cudaStream_t s) { spmv_launch<SPMV_ADD, T>(A, x, nullptr, nullptr, 0, y, s); }
template <class T> void launch_residual(SellViewT<T> A, const T* x, const T* b, T* r, cudaStream_t s) { spmv_launch<SPMV_RESID, T>(A, x, b, nullptr, 0, r, s); }
template <class T> void launch_jacobi(SellViewT<T> A, const T* dinv, const T* b, const T* x, T* x_out, double omega, cudaStream_t s) {
  spmv_launch<SPMV_JACOBI, T>(A, x, b, dinv, omega, x_out, s);
}
#define SHAKTI_INSTANTIATE_SPMV(T)                                                                       \
  template void launch_spmv<T>(SellViewT<T>, const T*, T*, cudaStream_t);                                \
  template void launch_spmv_add<T>(SellViewT<T>, const T*, T*, cudaStream_t);                            \
  template void launch_residual<T>(SellViewT<T>, const T*, const T*, T*, cudaStream_t);                  \
  template void launch_jacobi<T>(SellViewT<T>, const T*, const T*, const T*, T*, double, cudaStream_t);
SHAKTI_INSTANTIATE_SPMV(double)
SHAKTI_INSTANTIATE_SPMV(float)

__global__ void d2f_kernel(int64_t n, const double* __restrict__ a, float* __restrict__ out) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) out[i] = (float)a[i];
}
__global__ void f2d_kernel(int64_t n, const float* __restrict__ a, double* __restrict__ out) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) out[i] = (double)a[i];
}
static int stream_blocks(int64_t n) { return (int)std::min<int64_t>(148 * 16, std::max<int64_t>(1, (n + 255) / 256)); }
void launch_d2f(int64_t n, const double* a, float* out, cudaStream_t s) {
  if (n == 0) return;
  SHAKTI_LAUNCH(d2f_kernel, stream_blocks(n), 256, 0, s, n, a, out);
}
void launch_f2d(int64_t n, const float* a, double* out, cudaStream_t s) {
  if (n == 0) return;
  SHAKTI_LAUNCH(f2d_kernel, stream_blocks(n), 256, 0, s, n, a, out);
}
__global__ void __launch_bounds__(256)
sell_scale_to_half_kernel(SellView A, const double* __restrict__ dinv, __half* __restrict__ out) {
  const int32_t row = blockIdx.x * blockDim.x + threadIdx.x;
  const int32_t slice = row >> 5;
  if (slice >= A.n_slices) return;
  const int32_t base = A.slice_ptr[slice] + (row & 31);
  const int32_t w = (A.slice_ptr[slice + 1] - A.slice_ptr[slice]) >> 5;
  const double s = row < A.n_rows ? dinv[row] : 0.0;
  for (int k = 0; k < w; ++k) out[base + 32 * k] = __float2half_rn((float)(s * A.val[base + 32 * k]));
}
void DevSell::refresh_f16_scaled(const double* dinv, cudaStream_t s) const {
  if (valh.n != (size_t)padded) valh.alloc((size_t)std::max<int64_t>(padded, 1));
  if (n_rows == 0) return;
  SHAKTI_LAUNCH(sell_scale_to_half_kernel, div_up((int64_t)n_slices * 32, 256), 256, 0, s, view(*this), dinv, valh.p);
}
void DevSell::refresh_f32(cudaStream_t s) const {
  if (valf.n != (size_t)padded) valf.alloc((size_t)padded);
  launch_d2f(padded, val.p, valf.p, s);
}
template <class T>
__global__ void scaled_mul_kernel(int64_t n, const T* __restrict__ a, const T* __restrict__ b, T scale, T* __restrict__ out) {
  pdl_sync();
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) out[i] = scale * a[i] * b[i];
}
template <class T> void launch_scaled_mul(int64_t n, const T* a, const T* b, double scale, T* out, cudaStream_t s) {
  if (n == 0) return;
  SHAKTI_LAUNCH((scaled_mul_kernel<T>), stream_blocks(n), 256, 0, s, n, a, b, (T)scale, out);
}
template void launch_scaled_mul<double>(int64_t, const double*, const double*, double, double*, cudaStream_t);
template void launch_scaled_mul<float>(int64_t, const float*, const float*, double, float*, cudaStream_t);
template <class T>
__global__ void fill_t_kernel(int64_t n, T v, T* __restrict__ x) {
  pdl_sync();
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) x[i] = v;
}
template <class T> void launch_fill_t(int64_t n, T v, T* x, cudaStream_t s) {
  if (n == 0) return;
  SHAKTI_LAUNCH((fill_t_kernel<T>), stream_blocks(n), 256, 0, s, n, v, x);
}
template void launch_fill_t<double>(int64_t, double, double*, cudaStream_t);
template void launch_fill_t<float>(int64_t, float, float*, cudaStream_t);

__global__ void extract_dinv_kernel(int32_t n, const int32_t* __restrict__ diag_pos, const double* __restrict__ val,
                                    double* __restrict__ dinv) {
  const int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double d = val[diag_pos[i]];
  dinv[i] = d != 0.0 ? 1.0 / d : 1.0;
}
void launch_extract_dinv(int32_t n, const int32_t* diag_pos, const double* val, double* dinv, cudaStream_t s) {
  if (n == 0) return;
  SHAKTI_LAUNCH(extract_dinv_kernel, div_up(n, 256), 256, 0, s, n, diag_pos, val, dinv);
}

// ------------------------------------------------------------------ reductions
constexpr int kRedThreads = 256;

void Reducer::init(int sm_count) {
  max_blocks = sm_count * 8;
  partial.alloc((size_t)max_blocks * 32);
  counter.alloc_zero(1);
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// out[k] = sum_i V[k*ld + i] * w[i], k < NV.  Two stages in one launch: per-block partials,
// then the last block to finish sums them in a fixed order (deterministic result).
template <int NV>
__global__ void __launch_bounds__(kRedThreads)
multi_dot_kernel(int64_t n, const double* __restrict__ V, int64_t ld, const double* __restrict__ w,
                 double* __restrict__ partial, unsigned int* __restrict__ counter, double* __restrict__ out) {
  double acc[NV];
#pragma unroll
  for (int k = 0; k < NV; ++k) acc[k] = 0.0;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const double wi = w[i];
#pragma unroll
    for (int k = 0; k < NV; ++k) acc[k] += V[k * ld + i] * wi;
  }
  __shared__ double sm[NV][kRedThreads / 32];
  __shared__ bool is_last;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    const double v = warp_sum(acc[k]);
    if (lane == 0) sm[k][wid] = v;
  }
  __syncthreads();
  if (threadIdx.x < NV) {
    double v = 0.0;
#pragma unroll
    for (int j = 0; j < kRedThreads / 32; ++j) v += sm[threadIdx.x][j];
    partial[(size_t)blockIdx.x * NV + threadIdx.x] = v;
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) is_last = (atomicAdd(counter, 1u) == gridDim.x - 1);
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  for (int k = wid; k < NV; k += kRedThreads / 32) {
    double v = 0.0;
    for (int b = lane; b < (int)gridDim.x; b += 32) v += partial[(size_t)b * NV + k];
    v = warp_sum(v);
    if (lane == 0) out[k] = v;
  }
  if (threadIdx.x == 0) *counter = 0u;
}

void launch_multi_dot(Reducer& red, int64_t n, int nvec, const double* V, int64_t ld, const double* w,
                      double* out, cudaStream_t s) {
  int blocks = (int)std::min<int64_t>(red.max_blocks, std::max<int64_t>(1, (n + kRedThreads * 4 - 1) / (kRedThreads * 4)));
  int done = 0;
  while (done < nvec) {
    const int c = std::min(8, nvec - done);
    const double* Vc = V + (int64_t)done * ld;
    double* oc = out + done;
    switch (c) {
      case 1: SHAKTI_LAUNCH(multi_dot_kernel<1>, blocks, kRedThreads, 0, s, n, Vc, ld, w, red.partial.p, red.counter.p, oc); break;
      case 2: SHAKTI_LAUNCH(multi_dot_kernel<2>, blocks, kRedThreads, 0, s, n, Vc, ld, w, red.partial.p, red.counter.p, oc); break;
      case 3: SHAKTI_LAUNCH(multi_dot_kernel<3>, blocks, kRedThreads, 0, s, n, Vc, ld, w, red.partial.p, red.counter.p, oc); break;
      case 4: SHAKTI_LAUNCH(multi_dot_kernel<4>, blocks, kRedThreads, 0, s, n, Vc, ld, w, red.partial.p, red.counter.p, oc); break;
      case 5: SHAKTI_LAUNCH(multi_dot_kernel<5>, blocks, kRedThreads, 0, s, n, Vc, ld, w, red.partial.p, red.counter.p, oc); break;
      case 6: SHAKTI_LAUNCH(multi_dot_kernel<6>, blocks, kRedThreads, 0, s, n, Vc, ld, w, red.partial.p, red.counter.p, oc); break;
      case 7: SHAKTI_LAUNCH(multi_dot_kernel<7>, blocks, kRedThreads, 0, s, n, Vc, ld, w, red.partial.p, red.counter.p, oc); break;
      default: SHAKTI_LAUNCH(multi_dot_kernel<8>, blocks, kRedThreads, 0, s, n, Vc, ld, w, red.partial.p, red.counter.p, oc); break;
    }
    done += c;
  }
}

// Second classical Gram-Schmidt pass fused with the first pass's update:
//   w <- w - sum_k h[k] V_k ;  out[k] = <V_k, w_new> (k < nvec) ;  out[nvec] = <w_new, w_new>
// The basis is read once for both.  nvec <= NV; deterministic two-stage reduction as in multi_dot.
template <int NV>
__global__ void __launch_bounds__(kRedThreads)
orth_update_dot_kernel(int64_t n, int nvec, const double* __restrict__ V, int64_t ld, const double* __restrict__ h,
                       double* __restrict__ w, double* __restrict__ partial, unsigned int* __restrict__ counter,
                       double* __restrict__ out) {
  double hk[NV], acc[NV + 1];
#pragma unroll
  for (int k = 0; k < NV; ++k) { hk[k] = k < nvec ? h[k] : 0.0; acc[k] = 0.0; }
  acc[NV] = 0.0;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    double vk[NV];
    double a = 0.0;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      vk[k] = k < nvec ? V[k * ld + i] : 0.0;
      a += hk[k] * vk[k];
    }
    const double wn = w[i] - a;
    w[i] = wn;
#pragma unroll
    for (int k = 0; k < NV; ++k) acc[k] += vk[k] * wn;
    acc[NV] += wn * wn;
  }
  __shared__ double sm[NV + 1][kRedThreads / 32];
  __shared__ bool is_last;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k <= NV; ++k) {
    const double v = warp_sum(acc[k]);
    if (lane == 0) sm[k][wid] = v;
  }
  __syncthreads();
  if (threadIdx.x <= NV) {
    double v = 0.0;
#pragma unroll
    for (int j = 0; j < kRedThreads / 32; ++j) v += sm[threadIdx.x][j];
    partial[(size_t)blockIdx.x * (NV + 1) + threadIdx.x] = v;
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) is_last = (atomicAdd(counter, 1u) == gridDim.x - 1);
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  for (int k = wid; k <= NV; k += kRedThreads / 32) {
    double v = 0.0;
    for (int b = lane; b < (int)gridDim.x; b += 32) v += partial[(size_t)b * (NV + 1) + k];
    v = warp_sum(v);
    if (lane == 0) {
      if (k < nvec) out[k] = v;
      else if (k == NV) out[nvec] = v;
    }
  }
  if (threadIdx.x == 0) *counter = 0u;
}

// returns false if nvec is too large for the fused kernel (caller falls back to separate passes)
bool launch_orth_update_dot(Reducer& red, int64_t n, int nvec, const double* V, int64_t ld, const double* h, double* w,
                            double* out, cudaStream_t s) {
  if (nvec > 24) return false;
  const int blocks = (int)std::min<int64_t>(red.max_blocks, std::max<int64_t>(1, (n + kRedThreads * 4 - 1) / (kRedThreads * 4)));
  if (nvec <= 8) SHAKTI_LAUNCH(orth_update_dot_kernel<8>, blocks, kRedThreads, 0, s, n, nvec, V, ld, h, w, red.partial.p, red.counter.p, out);
  else if (nvec <= 16) SHAKTI_LAUNCH(orth_update_dot_kernel<16>, blocks, kRedThreads, 0, s, n, nvec, V, ld, h, w, red.partial.p, red.counter.p, out);
  else SHAKTI_LAUNCH(orth_update_dot_kernel<24>, blocks, kRedThreads, 0, s, n, nvec, V, ld, h, w, red.partial.p, red.counter.p, out);
  return true;
}

// w -= sum_k h[k] V_k  (SUB) or y = sum_k h[k] V_k (SET, first chunk) / y += ... (ADD)
enum { COMB_SUB = 0, COMB_SET = 1, COMB_ADD = 2, COMB_SUB_SCALE = 3 };
template <int NV, int MODE>
__global__ void __launch_bounds__(256)
combine_kernel(int64_t n, const double* __restrict__ V, int64_t ld, const double* __restrict__ h,
               double* __restrict__ w, double scale) {
  double hk[NV];
#pragma unroll
  for (int k = 0; k < NV; ++k) hk[k] = h[k];
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    double acc = 0.0;
#pragma unroll
    for (int k = 0; k < NV; ++k) acc += hk[k] * V[k * ld + i];
    if (MODE == COMB_SUB) w[i] -= acc;
    else if (MODE == COMB_SET) w[i] = acc;
    else if (MODE == COMB_ADD) w[i] += acc;
    else w[i] = (w[i] - acc) * scale;
  }
}

template <int MODE>
static void combine_chunk(int c, int blocks, int64_t n, const double* V, int64_t ld, const double* h, double* w,
                          cudaStream_t s, double scale = 1.0) {
  switch (c) {
    case 1: SHAKTI_LAUNCH((combine_kernel<1, MODE>), blocks, 256, 0, s, n, V, ld, h, w, scale); break;
    case 2: SHAKTI_LAUNCH((combine_kernel<2, MODE>), blocks, 256, 0, s, n, V, ld, h, w, scale); break;
    case 3: SHAKTI_LAUNCH((combine_kernel<3, MODE>), blocks, 256, 0, s, n, V, ld, h, w, scale); break;
    case 4: SHAKTI_LAUNCH((combine_kernel<4, MODE>), blocks, 256, 0, s, n, V, ld, h, w, scale); break;
    case 5: SHAKTI_LAUNCH((combine_kernel<5, MODE>), blocks, 256, 0, s, n, V, ld, h, w, scale); break;
    case 6: SHAKTI_LAUNCH((combine_kernel<6, MODE>), blocks, 256, 0, s, n, V, ld, h, w, scale); break;
    case 7: SHAKTI_LAUNCH((combine_kernel<7, MODE>), blocks, 256, 0, s, n, V, ld, h, w, scale); break;
    default: SHAKTI_LAUNCH((combine_kernel<8, MODE>), blocks, 256, 0, s, n, V, ld, h, w, scale); break;
  }
}

void launch_multi_axpy_neg(int64_t n, int nvec, const double* V, int64_t ld, const double* h, double* w,
                           cudaStream_t s) {
  if (n == 0) return;
  for (int done = 0; done < nvec; done += 8)
    combine_chunk<COMB_SUB>(std::min(8, nvec - done), stream_blocks(n), n, V + (int64_t)done * ld, ld, h + done, w, s);
}
// w = (w - sum_k h[k] V_k) * scale : Gram-Schmidt update fused with the normalisation
void launch_multi_axpy_neg_scale(int64_t n, int nvec, const double* V, int64_t ld, const double* h, double* w, double scale,
                                 cudaStream_t s) {
  if (n == 0) return;
  for (int done = 0; done < nvec; done += 8) {
    const int c = std::min(8, nvec - done);
    if (done + c >= nvec) combine_chunk<COMB_SUB_SCALE>(c, stream_blocks(n), n, V + (int64_t)done * ld, ld, h + done, w, s, scale);
    else combine_chunk<COMB_SUB>(c, stream_blocks(n), n, V + (int64_t)done * ld, ld, h + done, w, s);
  }
}
void launch_combine(int64_t n, int nvec, const double* V, int64_t ld, const double* h, double* y, cudaStream_t s) {
  if (n == 0) return;
  for (int done = 0; done < nvec; done += 8) {
    const int c = std::min(8, nvec - done);
    if (done == 0) combine_chunk<COMB_SET>(c, stream_blocks(n), n, V, ld, h, y, s);
    else combine_chunk<COMB_ADD>(c, stream_blocks(n), n, V + (int64_t)done * ld, ld, h + done, y, s);
  }
}

__global__ void readback_kernel(const double* __restrict__ src, double* __restrict__ dst_host, int count) {
  for (int i = threadIdx.x; i < count; i += blockDim.x) dst_host[i] = src[i];
  __threadfence_system();
}
void launch_readback(const double* src, double* dst_host, int count, cudaStream_t s) {
  if (count <= 0) return;
  SHAKTI_LAUNCH(readback_kernel, 1, 64, 0, s, src, dst_host, count);
}

// ------------------------------------------------------------------ model_setup data ingestion (SURVEY row f3)
// Bilinear interpolation of a gridded field f[iy][ix] (row-major, grid axes xg / yg ascending, not
// necessarily uniform) at scattered points, linear EXTRAPOLATION outside the grid: the semantics of
// scipy RegularGridInterpolator((x, y), f.T, bounds_error=False, fill_value=None), which the reference
// uses to bring BedMachine / ATL14 rasters onto the mesh nodes (model_setup.py:74-91).
__device__ __forceinline__ int grid_interval(const double* __restrict__ g, int n, double v) {
  int lo = 0, hi = n;              // first index with g[idx] > v  (searchsorted right) ...
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (g[mid] <= v) lo = mid + 1; else hi = mid;
  }
  return min(max(lo - 1, 0), n - 2);   // ... minus one, clipped so that [i, i+1] is a valid cell
}
__global__ void __launch_bounds__(256)
interp_grid_kernel(int64_t n, const double* __restrict__ px, const double* __restrict__ py, int nx, int ny,
                   const double* __restrict__ xg, const double* __restrict__ yg, const double* __restrict__ f,
                   double* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double x = px[i], y = py[i];
  const int ix = grid_interval(xg, nx, x), iy = grid_interval(yg, ny, y);
  const double tx = (x - xg[ix]) / (xg[ix + 1] - xg[ix]);
  const double ty = (y - yg[iy]) / (yg[iy + 1] - yg[iy]);
  const double f00 = f[(size_t)iy * nx + ix], f10 = f[(size_t)iy * nx + ix + 1];
  const double f01 = f[(size_t)(iy + 1) * nx + ix], f11 = f[(size_t)(iy + 1) * nx + ix + 1];
  out[i] = (1.0 - tx) * (1.0 - ty) * f00 + tx * (1.0 - ty) * f10 + (1.0 - tx) * ty * f01 + tx * ty * f11;
}
void launch_interp_grid(int64_t n, const double* px, const double* py, int nx, int ny, const double* xg, const double* yg,
                        const double* f, double* out, cudaStream_t s) {
  if (n == 0) return;
  SHAKTI_LAUNCH(interp_grid_kernel, div_up(n, 256), 256, 0, s, n, px, py, nx, ny, xg, yg, f, out);
}

// Lake indicator: even-odd rule against a closed polygon (vertices in shared memory, 1024 per pass); what
// set_lake_bdry does point by point with shapely in the reference (model_setup.py:68-72).
__global__ void __launch_bounds__(256)
points_in_polygon_kernel(int64_t n, const double* __restrict__ px, const double* __restrict__ py, int m,
                         const double* __restrict__ poly, double* __restrict__ out) {
  __shared__ double sx[1025], sy[1025];
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const double x = i < n ? px[i] : 0.0, y = i < n ? py[i] : 0.0;
  bool inside = false;
  for (int base = 0; base < m; base += 1024) {
    const int cnt = min(1024, m - base);
    __syncthreads();
    for (int k = threadIdx.x; k <= cnt; k += blockDim.x) {   // one extra vertex: the edge's end point
      const int v = (base + k) % m;
      sx[k] = poly[2 * v];
      sy[k] = poly[2 * v + 1];
    }
    __syncthreads();
    for (int k = 0; k < cnt; ++k) {
      const double x0 = sx[k], y0 = sy[k], x1 = sx[k + 1], y1 = sy[k + 1];
      if ((y0 > y) != (y1 > y)) {
        const double xc = x0 + (y - y0) * (x1 - x0) / (y1 - y0);
        if (x < xc) inside = !inside;
      }
    }
  }
  if (i < n) out[i] = inside ? 1.0 : 0.0;
}
void launch_points_in_polygon(int64_t n, const double* px, const double* py, int m, const double* poly, double* out,
                              cudaStream_t s) {
  if (n == 0) return;
  SHAKTI_LAUNCH(points_in_polygon_kernel, div_up(n, 256), 256, 0, s, n, px, py, m, poly, out);
}

// ------------------------------------------------------------------ streaming vector kernels
__global__ void axpy_kernel(int64_t n, double alpha, const double* __restrict__ x, double* __restrict__ y) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) y[i] += alpha * x[i];
}
void launch_axpy(int64_t n, double alpha, const double* x, double* y, cudaStream_t s) {
  if (n == 0) return;
  SHAKTI_LAUNCH(axpy_kernel, stream_blocks(n), 256, 0, s, n, alpha, x, y);
}
// out = mask ? 0 : a
__global__ void xmy_masked_kernel(int64_t n, const double* __restrict__ a, const uint8_t* __restrict__ mask,
                                  double* __restrict__ out) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) out[i] = mask[i] ? 0.0 : a[i];
}
void launch_xmy_masked(int64_t n, const double* a, const uint8_t* mask, double* out, cudaStream_t s) {
  if (n == 0) return;
  SHAKTI_LAUNCH(xmy_masked_kernel, stream_blocks(n), 256, 0, s, n, a, mask, out);
}
__global__ void gather_kernel(int64_t n, const int32_t* __restrict__ idx, const double* __restrict__ src,
                              double* __restrict__ dst) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) dst[i] = src[idx[i]];
}
void launch_gather(int64_t n, const int32_t* idx, const double* src, double* dst, cudaStream_t s) {
  if (n == 0) return;
  SHAKTI_LAUNCH(gather_kernel, stream_blocks(n), 256, 0, s, n, idx, src, dst);
}
__global__ void scatter_kernel(int64_t n, const int32_t* __restrict__ idx, const double* __restrict__ src,
                               double* __restrict__ dst) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) dst[idx[i]] = src[i];
}
void launch_scatter(int64_t n, const int32_t* idx, const double* src, double* dst, cudaStream_t s) {
  if (n == 0) return;
  SHAKTI_LAUNCH(scatter_kernel, stream_blocks(n), 256, 0, s, n, idx, src, dst);
}
// static part of Head (constitutive.py:6-9): h0 = z_b + (rho_i/rho_w)(z_s - z_b)
__global__ void head0_kernel(int64_t n, const double* __restrict__ z_b, const double* __restrict__ z_s, double ratio,
                             double* __restrict__ h0) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    h0[i] = z_b[i] + ratio * (z_s[i] - z_b[i]);
}
void launch_head0(int64_t n, const double* z_b, const double* z_s, double ratio, double* h0, cudaStream_t s) {
  if (n == 0) return;
  SHAKTI_LAUNCH(head0_kernel, stream_blocks(n), 256, 0, s, n, z_b, z_s, ratio, h0);
}
__global__ void interleave_kernel(int64_t n, const double* __restrict__ a, const double* __restrict__ b,
                                  double* __restrict__ ab) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    ab[2 * i] = a[i];
    ab[2 * i + 1] = b[i];
  }
}
void launch_interleave(int64_t n, const double* a, const double* b, double* ab, cudaStream_t s) {
  if (n == 0) return;
  SHAKTI_LAUNCH(interleave_kernel, stream_blocks(n), 256, 0, s, n, a, b, ab);
}
__global__ void deinterleave_kernel(int64_t n, const double* __restrict__ ab, double* __restrict__ a,
                                    double* __restrict__ b) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    a[i] = ab[2 * i];
    b[i] = ab[2 * i + 1];
  }
}
void launch_deinterleave(int64_t n, const double* ab, double* a, double* b, cudaStream_t s) {
  if (n == 0) return;
  SHAKTI_LAUNCH(deinterleave_kernel, stream_blocks(n), 256, 0, s, n, ab, a, b);
}

// ------------------------------------------------------------------ water-budget diagnostics
// One record of the global water budget at the current state (DESIGN.md "Water-budget diagnostics").  Stage 1:
// every cell this rank counts (cell_counted) adds its unconstrained element residual F_a (element_core, no
// lifting) to the outflow (Dirichlet vertex, negated) or to the imbalance (other vertex), its source integrals
// by the assembly's own rules and its vertex extrema; each block reduces its threads in a fixed tree and
// writes one partial.  Stage 2: one block sums the partials in a fixed order.  No floating-point atomics, so
// a record is bitwise reproducible for a given grid.
constexpr int kDiagThreads = 256;

__device__ __forceinline__ void diag_block_reduce(double (&v)[kDiagVals], double* __restrict__ sh, double* __restrict__ out) {
  // sh: kDiagVals x kDiagThreads; sums for [0, kDiagSums), maxima after
#pragma unroll
  for (int k = 0; k < kDiagVals; ++k) sh[k * kDiagThreads + threadIdx.x] = v[k];
  __syncthreads();
  for (int w = kDiagThreads / 2; w > 0; w >>= 1) {
    if ((int)threadIdx.x < w) {
#pragma unroll
      for (int k = 0; k < kDiagVals; ++k) {
        const double a = sh[k * kDiagThreads + threadIdx.x], b = sh[k * kDiagThreads + threadIdx.x + w];
        sh[k * kDiagThreads + threadIdx.x] = k < kDiagSums ? a + b : fmax(a, b);
      }
    }
    __syncthreads();
  }
  if (threadIdx.x < kDiagVals) out[threadIdx.x] = sh[threadIdx.x * kDiagThreads];
}

__global__ void __launch_bounds__(kDiagThreads)
diagnostics_kernel(int32_t ne, const int32_t* __restrict__ c0, const int32_t* __restrict__ c1, const int32_t* __restrict__ c2,
                   const uint8_t* __restrict__ counted, FieldPtrs f, const double* __restrict__ kbar, double dt, DevParams p,
                   double* __restrict__ partial) {
  __shared__ double sh[kDiagVals * kDiagThreads];
  double v[kDiagVals];
#pragma unroll
  for (int k = 0; k < kDiagVals; ++k) v[k] = k < kDiagSums ? 0.0 : -INFINITY;
  const int32_t stride = gridDim.x * blockDim.x;
  for (int32_t e = blockIdx.x * blockDim.x + threadIdx.x; e < ne; e += stride) {
    if (!counted[e]) continue;
    const int32_t vv[3] = {c0[e], c1[e], c2[e]};
    const Geo g = geometry(f.x[vv[0]], f.y[vv[0]], f.x[vv[1]], f.y[vv[1]], f.x[vv[2]], f.y[vv[2]]);
    double h[3], bb[3], mm[3], qxv[3], qyv[3], Nv[3], Nn[3], st[3], Gv[3], inp[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      Nv[i] = f.N[vv[i]];
      h[i] = f.h0[vv[i]] - Nv[i] * p.inv_rwg;
      bb[i] = f.b[vv[i]];
      mm[i] = f.melt[vv[i]];
      qxv[i] = f.qx[vv[i]];
      qyv[i] = f.qy[vv[i]];
      Nn[i] = f.N_n[vv[i]];
      st[i] = f.storage[vv[i]];
      Gv[i] = f.G[vv[i]];
      inp[i] = f.inputs[vv[i]];
    }
    ElemOut o;
    element_core(g, h, bb, mm, qxv, qyv, Nv, Nn, st, Gv, inp, kbar[e], dt, p, o);
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      if (f.isbc[vv[a]]) v[kDiagOutflow] -= o.F[a];
      else v[kDiagImbalance] += o.F[a];
    }
    // melt m0 + mdiff at the vertices, as element_core forms it (constitutive.py:25-26)
    double ghx = 0, ghy = 0, gbx = 0, gby = 0, gmx = 0, gmy = 0;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      ghx += h[i] * g.gx[i];  ghy += h[i] * g.gy[i];
      gbx += bb[i] * g.gx[i]; gby += bb[i] * g.gy[i];
      gmx += mm[i] * g.gx[i]; gmy += mm[i] * g.gy[i];
    }
    const double gb2 = gbx * gbx + gby * gby, gmgb = gmx * gbx + gmy * gby, inv1 = 1.0 / (1.0 + gb2);
    double smelt = 0, sinp = 0, sb = 0, sN = 0, ss = 0, sd = 0, ssd = 0;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      smelt += (Gv[i] - p.rwg * (qxv[i] * ghx + qyv[i] * ghy)) * p.inv_Lh + (gb2 * mm[i] + bb[i] * gmgb) * inv1;
      sinp += inp[i];
      sb += bb[i];
      sN += Nv[i];
      const double d = Nv[i] - Nn[i];
      ss += st[i];
      sd += d;
      ssd += st[i] * d;
    }
    const double m6 = g.detabs * (1.0 / 6.0);   // int phi_a = |detJ| / 6
    v[kDiagArea] += 0.5 * g.detabs;
    v[kDiagVolume] += m6 * sb;
    v[kDiagInput] += m6 * sinp;
    v[kDiagMelt] += m6 * smelt;
    v[kDiagIntN] += m6 * sN;
    // storage: int s (N - N_n) of two P1 functions, times 1/(rho_w g dt)
    v[kDiagStorage] += p.inv_rwg / dt * g.detabs * (1.0 / 24.0) * (ss * sd + ssd);
    // closure A b N|N|^(n-1) by the assembly's rule: Radon-7 for n = 3, the __constant__ table otherwise
    double clos = 0;
    if (p.n_is_3) {
      double f0, f1, f2, m00, m01, m02, m11, m12, m22;
      reaction_radon7<false>(g.detabs, bb, Nv, Nn, st, 0.0, p.A, f0, f1, f2, m00, m01, m02, m11, m12, m22);
      clos = f0 + f1 + f2;
    } else {
      const double e1 = p.n - 1.0;
      const int nq = c_nrq;
      for (int k = 0; k < nq; ++k) {
        const double l0 = c_rq[4 * k], l1 = c_rq[4 * k + 1], l2 = c_rq[4 * k + 2];
        const double bq = l0 * bb[0] + l1 * bb[1] + l2 * bb[2];
        const double Nq = l0 * Nv[0] + l1 * Nv[1] + l2 * Nv[2];
        clos += c_rq[4 * k + 3] * g.detabs * (p.A * bq * Nq * pow(fabs(Nq), e1));
      }
    }
    v[kDiagClosure] += clos;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      v[kDiagNegNmin] = fmax(v[kDiagNegNmin], -Nv[i]);
      v[kDiagNmax] = fmax(v[kDiagNmax], Nv[i]);
      v[kDiagBmax] = fmax(v[kDiagBmax], bb[i]);
    }
  }
  diag_block_reduce(v, sh, partial + (size_t)blockIdx.x * kDiagVals);
}

// global values vals[kDiagVals] -> one record row[SHAKTI_D_COUNT]
__device__ __forceinline__ void diag_write_row(const double* vals, double* row, double dt, double its, double residual) {
  row[SHAKTI_D_DT] = dt;
  row[SHAKTI_D_NEWTON_ITS] = its;
  row[SHAKTI_D_RESIDUAL] = residual;
#pragma unroll
  for (int k = 0; k <= kDiagImbalance; ++k) row[SHAKTI_D_AREA + k] = vals[k];
  row[SHAKTI_D_N_MEAN] = vals[kDiagIntN] / vals[kDiagArea];
  row[SHAKTI_D_N_MIN] = -vals[kDiagNegNmin];
  row[SHAKTI_D_N_MAX] = vals[kDiagNmax];
  row[SHAKTI_D_B_MAX] = vals[kDiagBmax];
}

__global__ void __launch_bounds__(kDiagThreads)
diagnostics_finish_kernel(int nparts, const double* __restrict__ partial, double* __restrict__ vals, double* __restrict__ row,
                          double dt, double its, double residual) {
  __shared__ double sh[kDiagVals * kDiagThreads];
  double v[kDiagVals];
#pragma unroll
  for (int k = 0; k < kDiagVals; ++k) v[k] = k < kDiagSums ? 0.0 : -INFINITY;
  for (int b = threadIdx.x; b < nparts; b += kDiagThreads)
#pragma unroll
    for (int k = 0; k < kDiagVals; ++k) v[k] = k < kDiagSums ? v[k] + partial[(size_t)b * kDiagVals + k] : fmax(v[k], partial[(size_t)b * kDiagVals + k]);
  diag_block_reduce(v, sh, vals);
  if (row == nullptr) return;
  __syncthreads();
  if (threadIdx.x == 0) diag_write_row(vals, row, dt, its, residual);
}

__global__ void diagnostics_row_kernel(const double* __restrict__ vals, double* __restrict__ row, double dt, double its,
                                       double residual) {
  diag_write_row(vals, row, dt, its, residual);
}

int diagnostics_parts(int32_t ne, int sm_count) { return std::max(1, std::min(div_up(ne, kDiagThreads), 4 * sm_count)); }

void launch_diagnostics(int32_t ne, const int32_t* c0, const int32_t* c1, const int32_t* c2, const uint8_t* counted, FieldPtrs f,
                        const double* kbar, double dt, DevParams p, int nparts, double* partial, double* vals, double* row,
                        double its, double residual, cudaStream_t s) {
  if (ne > 0) SHAKTI_LAUNCH(diagnostics_kernel, nparts, kDiagThreads, 0, s, ne, c0, c1, c2, counted, f, kbar, dt, p, partial);
  SHAKTI_LAUNCH(diagnostics_finish_kernel, 1, kDiagThreads, 0, s, ne > 0 ? nparts : 0, partial, vals, row, dt, its, residual);
}

void launch_diagnostics_row(const double* vals, double* row, double dt, double its, double residual, cudaStream_t s) {
  SHAKTI_LAUNCH(diagnostics_row_kernel, 1, 1, 0, s, vals, row, dt, its, residual);
}

}  // namespace shakti
