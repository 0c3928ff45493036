// C ABI of the B200-native SHAKTI solver (include/shakti_b200.h): the model object, the
// Newton loop, the time step and the parity hooks.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <memory>

#include "amg.h"
#include "comm.h"
#include "device.h"
#include "krylov.h"

namespace shakti {

static thread_local std::string t_last_error;
void set_last_error(const std::string& msg) { t_last_error = msg; }

// default degree-7 table: collapsed Gauss-Jacobi 4x4, generated below by Golub-Welsch (stand-in for
// Basix' default; the CPU checker under tests/ builds the same rule independently and checks its degree)
static void default_k_rule(std::vector<double>& pts, std::vector<double>& wts);
}  // namespace shakti

using namespace shakti;

struct shakti_model {
  int device = 0;
  int sm_count = 148;
  cudaStream_t stream = nullptr;
  shakti_params prm;
  DevParams dprm;
  shakti_options opt;
  HostMesh hm;
  std::vector<int32_t> cells_g;   // caller cells (parity hooks, Dirichlet location)
  std::unique_ptr<HostCsr> csr_g; // caller CSR pattern, built lazily
  // quadrature
  std::vector<double> kq_pts, kq_wts;
  // device mesh
  DevBuf<double> x, y;
  DevBuf<int32_t> c0, c1, c2, slot, diag_pos, win, l2g;
  // row-block assembly plan (prep.h AssemblyBlocks)
  AssemblyBlocks ab;
  DevBuf<int32_t> ab_eptr, ab_elems, ab_incptr, ab_hptr, ab_halo;
  DevBuf<uint16_t> ab_inc, ab_lv;
  DevBuf<uint32_t> ab_src;
  // vertex fields (n_local)
  DevBuf<double> z_b, z_s, h0, G, inputs, storage, b, b2, N, N_n, qx, qy, melt, melt2, F, dx, rhs, dinv;
  DevBuf<double> kbar;
  DevBuf<uint8_t> isbc;
  DevBuf<double> stage;   // nv_g doubles: caller-numbered staging for set/get
  DevBuf<double> stage2;  // 2 nv_g (interleaved flux)
  DevBuf<double> scal;    // small device scalars
  double* host_scal = nullptr;  // pinned
  // asynchronous output path (shakti_step_host_async): snapshots of b, N, qx, qy taken on the compute
  // stream, copied to the caller's host buffers on a second stream while the next step runs
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t ev_snap = nullptr, ev_d2h = nullptr;
  DevBuf<double> out_stage[4];
  bool d2h_pending = false;
  // shakti_snapshot / shakti_rollback: device-side copy of the time-dependent state
  DevBuf<double> snap[6];
  double snap_hist_ratio = -1.0, snap_hist_dt = 0.0, snap_residual0 = 0.0;
  int64_t snap_steps = 0;
  bool snap_valid = false;
  // water-budget diagnostics: cells this rank counts, reduction scratch (partials; rank values + one-shot row)
  // and the record buffer of diag_cap rows, diag_n of them filled (snap_diag_n at the last snapshot)
  DevBuf<uint8_t> cell_counted;
  DevBuf<double> diag_partial, diag_vals, diag_rows;
  int diag_parts = 1;
  int64_t diag_cap = 0, diag_n = 0, snap_diag_n = 0;
  // model clock [s]: a solve with step dt is forced at t_model + dt; update_b advances it by dt
  double t_model = 0.0, snap_t_model = 0.0;
  // moulins (shakti_set_moulins): every moulin in caller order on the host (mo_kptr/mo_t/mo_q: CSR of the knots),
  // this rank's moulins on the device grouped by row (MoulinView), mo_own: their caller indices in that order
  int64_t n_moulins = 0;
  std::vector<int32_t> mo_vertex;
  std::vector<int64_t> mo_kptr;
  std::vector<double> mo_t, mo_q;
  double mo_period = 0.0;
  std::vector<int64_t> mo_own;
  int32_t mo_rows = 0;
  DevBuf<int32_t> mo_row_d, mo_rptr_d;
  DevBuf<int64_t> mo_kptr_d;
  DevBuf<double> mo_t_d, mo_q_d;
  std::vector<int32_t> bc_g;   // Dirichlet dofs (caller ids, sorted)
  double N_bdry = 0.0;
  int64_t n_bc = 0;
  bool h0_dirty = true;
  DevSell J;
  bool J_valid = false;
  HaloPlan halo;
  Gmres gmres;
  BiCgStab bicg;
  bool bicg_init = false;
  Reducer red;
  std::unique_ptr<Amg> amg;
  bool amg_setup_done = false;
  int64_t step_of_refresh = -1000000;  // st.steps at the last AMG refresh
  int newton_it_in_step = 0;           // Newton iteration index of the solve in progress
  double rate_after_refresh = 0.0;     // Krylov iterations per decade of the first solve after the last refresh
  double last_rate = 0.0;              // ... and of the latest solve
  // adaptive Krylov tolerance (linear_forcing): contraction r1/r0 of the previous time step's first
  // Newton iteration and the dt it was observed with (<= 0: nothing known)
  double hist_ratio = -1.0, hist_dt = 0.0;
  // Newton state
  double residual0 = 0.0;  // DOLFINx NewtonSolver::_residual0 (kept across solves)
  shakti_stats st{};
  int64_t launches_at_create = 0;

  FieldPtrs fields() const {
    FieldPtrs f;
    f.x = x.p; f.y = y.p; f.h0 = h0.p; f.N = N.p; f.N_n = N_n.p; f.b = b.p; f.qx = qx.p; f.qy = qy.p;
    f.G = G.p; f.melt = melt.p; f.storage = storage.p; f.inputs = inputs.p; f.isbc = isbc.p;
    return f;
  }
};

namespace shakti {

static void use_device(shakti_model* m) { SHAKTI_CUDA(cudaSetDevice(m->device)); }

static void refresh_h0(shakti_model* m) {
  if (!m->h0_dirty) return;
  launch_head0(m->hm.n_local, m->z_b.p, m->z_s.p, m->prm.rho_i / m->prm.rho_w, m->h0.p, m->stream);
  m->h0_dirty = false;
}

static double* field_ptr(shakti_model* m, int f) {
  switch (f) {
    case SHAKTI_F_Z_B: return m->z_b.p;
    case SHAKTI_F_Z_S: return m->z_s.p;
    case SHAKTI_F_G: return m->G.p;
    case SHAKTI_F_INPUTS: return m->inputs.p;
    case SHAKTI_F_STORAGE: return m->storage.p;
    case SHAKTI_F_B: return m->b.p;
    case SHAKTI_F_N: return m->N.p;
    case SHAKTI_F_N_N: return m->N_n.p;
    case SHAKTI_F_QX: return m->qx.p;
    case SHAKTI_F_QY: return m->qy.p;
    case SHAKTI_F_MELT_N: return m->melt.p;
    case SHAKTI_F_RESIDUAL: return m->F.p;
    default: throw Error(SHAKTI_ERR_INVALID, "unknown field id");
  }
}

// caller-numbered device array (nv_g) -> local field (n_local, ghosts included)
static void scatter_in(shakti_model* m, const double* src_dev, double* field) {
  launch_gather(m->hm.n_local, m->l2g.p, src_dev, field, m->stream);
}
// local field (owned part) -> caller-numbered device array; entries of other ranks are 0
static void gather_out(shakti_model* m, const double* field, double* dst_dev) {
  if (comm().active()) SHAKTI_CUDA(cudaMemsetAsync(dst_dev, 0, sizeof(double) * m->hm.nv_g, m->stream));
  launch_scatter(m->hm.n_owned, m->l2g.p, field, dst_dev, m->stream);
}

static void set_field(shakti_model* m, int f, const double* src, int is_device) {
  SHAKTI_REQUIRE(f >= 0 && f < SHAKTI_F_COUNT && f != SHAKTI_F_RESIDUAL, "field is not writable");
  SHAKTI_REQUIRE(src != nullptr, "null source");
  const double* s = src;
  if (!is_device) {
    SHAKTI_CUDA(cudaMemcpyAsync(m->stage.p, src, sizeof(double) * m->hm.nv_g, cudaMemcpyHostToDevice, m->stream));
    s = m->stage.p;
  }
  scatter_in(m, s, field_ptr(m, f));
  if (f == SHAKTI_F_Z_B || f == SHAKTI_F_Z_S) m->h0_dirty = true;
  if (f != SHAKTI_F_INPUTS) m->hist_ratio = -1.0;   // state replaced from outside: no convergence history
  if (!is_device) SHAKTI_CUDA(cudaStreamSynchronize(m->stream));
}

static void get_field(shakti_model* m, int f, double* dst, int is_device) {
  SHAKTI_REQUIRE(f >= 0 && f < SHAKTI_F_COUNT, "unknown field id");
  SHAKTI_REQUIRE(dst != nullptr, "null destination");
  if (is_device) {
    gather_out(m, field_ptr(m, f), dst);
  } else {
    gather_out(m, field_ptr(m, f), m->stage.p);
    SHAKTI_CUDA(cudaMemcpyAsync(dst, m->stage.p, sizeof(double) * m->hm.nv_g, cudaMemcpyDeviceToHost, m->stream));
    SHAKTI_CUDA(cudaStreamSynchronize(m->stream));
  }
}

static void allreduce(shakti_model* m, double* dev, int count) { comm_allreduce_sum(dev, count, m->stream); }

static double norm2(shakti_model* m, const double* v) {
  launch_multi_dot(m->red, m->hm.n_owned, 1, v, m->hm.n_owned, v, m->scal.p, m->stream);
  allreduce(m, m->scal.p, 1);
  launch_readback(m->scal.p, m->host_scal, 1, m->stream);
  SHAKTI_CUDA(cudaStreamSynchronize(m->stream));
  if (comm().p2p && p2p_error())
    throw Error(SHAKTI_ERR_COMM, "a peer-to-peer wait timed out (a rank of the job stopped responding)");
  return std::sqrt(std::max(m->host_scal[0], 0.0));
}

// The quadrature tables live in __constant__ memory, which is shared by all models of the process:
// a model re-uploads its own tables whenever another model used the kernels last.
static const shakti_model* g_rule_owner = nullptr;
static void ensure_rules(shakti_model* m) {
  if (g_rule_owner == m) return;
  upload_k_rule((int)m->kq_wts.size(), m->kq_pts.data(), m->kq_wts.data(), m->stream);
  if (!m->dprm.n_is_3) upload_reaction_rule((int)m->kq_wts.size(), m->kq_pts.data(), m->kq_wts.data(), m->stream);
  g_rule_owner = m;
}

static void compute_kbar(shakti_model* m) {
  SHAKTI_PHASE("kbar", m->stream);
  ensure_rules(m);
  launch_kbar(m->hm.ne, m->c0.p, m->c1.p, m->c2.p, m->x.p, m->y.p, m->b.p, m->qx.p, m->qy.p, m->kbar.p,
              m->dprm, m->stream);
}

static MoulinView moulin_view(const shakti_model* m) {
  return {m->mo_rows, m->mo_row_d.p, m->mo_rptr_d.p, m->mo_kptr_d.p, m->mo_t_d.p, m->mo_q_d.p, m->mo_period};
}

// F -= moulin discharge at the end of the step (t_model + dt).  Moulin rows are never Dirichlet rows, so this
// commutes with the Dirichlet replacement, and the Jacobian is unchanged.
static void apply_moulins(shakti_model* m, double dt) {
  if (m->n_moulins > 0) launch_moulin_source(moulin_view(m), m->t_model + dt, m->F.p, m->stream);
}

// total discharge of this rank's moulins at t, on the host (the same bits as the device evaluation)
static double owned_moulin_discharge(const shakti_model* m, double t) {
  double s = 0.0;
  for (int64_t k : m->mo_own) {
    const int64_t a = m->mo_kptr[k];
    s += hydrograph_at(m->mo_t.data() + a, m->mo_q.data() + a, m->mo_kptr[k + 1] - a, m->mo_period, t);
  }
  return s;
}

// residual (+ Jacobian) at the current state; Kbar must be current
static void assemble(shakti_model* m, double dt, int want_J) {
  SHAKTI_PHASE(want_J ? "assembleFJ" : "assembleF", m->stream);
  refresh_h0(m);
  ensure_rules(m);
  const int32_t no = m->hm.n_owned;
  if (m->opt.assembly_kernel == 0 && m->ab.ok) {
    AssemblyPlanView pl{no, m->ab.rows_per_block, m->ab.n_blocks, m->ab.max_cells, m->ab.max_verts, m->ab_eptr.p,
                        m->ab_elems.p, m->ab_lv.p, m->ab_hptr.p, m->ab_halo.p, m->ab_incptr.p, m->ab_inc.p, m->ab_src.p};
    launch_assemble_blocks(pl, m->fields(), m->kbar.p, dt, m->N_bdry, m->J.slice_ptr.p, m->F.p, m->J.val.p, want_J, m->dprm,
                           m->stream);
    apply_moulins(m, dt);
    if (want_J) m->J_valid = true;
    return;
  }
  SHAKTI_CUDA(cudaMemsetAsync(m->F.p, 0, sizeof(double) * no, m->stream));
  if (want_J) SHAKTI_CUDA(cudaMemsetAsync(m->J.val.p, 0, sizeof(double) * m->J.padded, m->stream));
  launch_assemble_atomic(m->hm.ne, no, m->c0.p, m->c1.p, m->c2.p, m->slot.p, m->fields(), m->kbar.p, dt,
                         m->N_bdry, m->F.p, m->J.val.p, want_J, m->dprm, m->stream);
  if (m->n_bc) launch_apply_bc(no, m->isbc.p, m->N.p, m->N_bdry, m->diag_pos.p, m->F.p, m->J.val.p, want_J, m->stream);
  apply_moulins(m, dt);
  if (want_J) m->J_valid = true;
}

static void ensure_amg(shakti_model* m) {
  if (m->amg_setup_done) return;
  AmgOptions ao;
  ao.max_levels = m->opt.amg_max_levels;
  ao.coarse_size = m->opt.amg_coarse_size;
  ao.presmooth = m->opt.amg_presmooth;
  ao.postsmooth = m->opt.amg_postsmooth;
  ao.smoother_omega = m->opt.amg_smoother_omega;
  ao.prolong_omega = m->opt.amg_prolong_omega;
  ao.strength_theta = m->opt.amg_strength_theta;
  ao.cheby_ratio = m->opt.amg_cheby_ratio;
  ao.smoother = m->opt.amg_smoother;
  ao.fp32_cycle = m->opt.amg_fp32_cycle;
  ao.smoother_halo = m->opt.amg_smoother_halo;
  ao.replicate_below = m->opt.amg_replicate_below;
  // The V-cycle is replayed as a CUDA graph on one GPU and, on several, when its halo exchanges and the
  // gather of the replicated level are our own P2P kernels (no NCCL call inside the cycle).  With NCCL
  // nodes in the graph the replay was slower than issuing them (round 1: 84 vs 70 ms/step on 8 B200s).
  ao.cuda_graph = m->opt.amg_cuda_graph && (!comm().active() || comm().p2p);
  std::vector<uint8_t> excl = m->isbc.download(m->stream);
  excl.resize(m->hm.n_owned);
  m->amg.reset(new Amg());
  m->amg->setup(m->hm.A, m->hm.S, excl, m->hm.nbrs, &m->halo, ao, m->sm_count, m->stream);
  m->amg_setup_done = true;
}

// Solve J dx = rhs (rhs, dx owned-length device vectors) with the configured method.
static KrylovResult linear_solve(shakti_model* m, const double* rhs, double* dx, double rtol) {
  SHAKTI_REQUIRE(m->J_valid, "no assembled Jacobian");
  const int32_t no = m->hm.n_owned;
  SellView Jv = view(m->J);
  ApplyFn A = [m, Jv](double* xl, double* y) {
    SHAKTI_PHASE("halo+spmv", m->stream);
    m->halo.exchange(xl, m->stream);
    launch_spmv(Jv, xl, y, m->stream);
  };
  AllReduceFn ar = [m](double* d, int c) { allreduce(m, d, c); };
  auto krylov = [&](const PrecFn& M, int max_it) {
    SHAKTI_PHASE("krylov_total", m->stream);
    if (m->opt.linear_solver == SHAKTI_KSP_BICGSTAB) {
      if (!m->bicg_init) { m->bicg.init(no, m->hm.n_local, m->sm_count, m->stream); m->bicg_init = true; }
      return m->bicg.solve(A, M, ar, rhs, dx, rtol, m->opt.linear_atol, max_it);
    }
    return m->gmres.solve(A, M, ar, rhs, dx, rtol, m->opt.linear_atol, max_it);
  };
  KrylovResult r;
  if (m->opt.precond == SHAKTI_PC_AMG) {
    ensure_amg(m);
    // The hierarchy is a preconditioner only: its numbers are recomputed at the first Newton
    // solve of every amg_refresh_every-th time step, or earlier when the Krylov iteration count
    // has grown by more than half since the last refresh.  The Krylov solve always uses the
    // current J, so a lagged hierarchy costs iterations, never accuracy; a solve that stalls on
    // a lagged hierarchy is repeated once with a fresh one.
    const int every = std::max(1, m->opt.amg_refresh_every);
    const bool due = m->newton_it_in_step == 0 && (m->st.steps - m->step_of_refresh) >= every;
    // iteration counts are compared per decade of residual reduction: the Krylov tolerance differs from
    // solve to solve (linear_forcing)
    const double decades = std::max(1.0, -std::log10(std::max(rtol, 1e-300)));
    const bool degraded = m->rate_after_refresh > 0 && m->last_rate > 1.5 * m->rate_after_refresh + 0.25;
    auto do_refresh = [&]() {
      SHAKTI_PHASE("amg_refresh", m->stream);
      m->amg->refresh(m->J, m->diag_pos.p);
      m->st.amg_refreshes++;
      m->step_of_refresh = m->st.steps;
      m->rate_after_refresh = -1.0;
    };
    bool fresh = false;
    if (!m->amg->ready() || due || degraded) { do_refresh(); fresh = true; }
    else { SHAKTI_PHASE("amg_fine_smoother", m->stream); m->amg->refresh_fine_smoother(m->J, m->diag_pos.p); }
    PrecFn M = [m](const double* rr, double* z) { SHAKTI_PHASE("vcycle", m->stream); m->amg->apply(m->J, rr, z); };
    int budget = m->opt.linear_max_it;
    if (!fresh && m->rate_after_refresh > 0) budget = std::min(budget, (int)(3.0 * m->rate_after_refresh * decades) + 20);
    r = krylov(M, budget);
    m->st.linear_its += r.iterations;
    if (!r.converged && !fresh) {
      do_refresh();
      r = krylov(M, m->opt.linear_max_it);
      m->st.linear_its += r.iterations;
    }
    m->last_rate = r.iterations / decades;
    if (m->rate_after_refresh < 0) m->rate_after_refresh = std::max(0.05, m->last_rate);
  } else {
    PrecFn M;
    if (m->opt.precond == SHAKTI_PC_JACOBI) {
      launch_extract_dinv(no, m->diag_pos.p, m->J.val.p, m->dinv.p, m->stream);
      M = [m, no](const double* rr, double* z) { launch_scaled_mul<double>(no, m->dinv.p, rr, 1.0, z, m->stream); };
    } else {
      M = [m, no](const double* rr, double* z) {
        SHAKTI_CUDA(cudaMemcpyAsync(z, rr, sizeof(double) * no, cudaMemcpyDeviceToDevice, m->stream));
      };
    }
    r = krylov(M, m->opt.linear_max_it);
    m->st.linear_its += r.iterations;
  }
  m->st.last_linear_relres = r.relres;
  return r;
}

// dx[bc] = F[bc]   (identity rows of J)
__global__ void fix_bc_dx_kernel(int32_t n, const uint8_t* __restrict__ isbc, const double* __restrict__ F,
                                 double* __restrict__ dx) {
  const int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && isbc[i]) dx[i] = F[i];
}

// DOLFINx NewtonSolver::solve (criterion "residual", relaxation 1, LU replaced by Krylov)
//
// The reference solves every Newton system exactly (LU).  Here the Krylov solve of Newton iteration k
// stops at an ABSOLUTE residual tau_k:
//   linear_forcing == 0 : tau_k = linear_rtol * ||F_0||            (F_0: residual the solve started from)
//   linear_forcing  > 0 : tau_k = max(linear_rtol ||F_0||, linear_forcing * pred_{k+1})  while another
//                         Newton iteration is expected to follow, and linear_rtol ||F_0|| for the solve that
//                         is expected to be the LAST one (pred_{k+1} within a decade of the Newton target)
// where pred_{k+1} is the residual an exact Newton step is expected to leave: the quadratic model
// r_k^3 / r_{k-1}^2 for k >= 1 and, for k = 0, the first contraction r_1/r_0 observed in the previous time
// step (same dt; nothing known => the tight tolerance).  With linear_forcing = 0.01 the inexactness
// changes the intermediate Newton residuals by ~1 % (errors of earlier iterates are damped quadratically)
// and the final iterate is solved as tightly as before, so the iteration counts and the converged fields
// are those of the exact iteration (tests: identical Newton counts, fields <= 1e-8 against the CPU LU
// restatement) at roughly 60 % of the Krylov iterations.
// One water-budget record of the current state into `row` (device, SHAKTI_D_COUNT doubles), on the stream.
// Kbar and h0 must be current.  With moulins, each rank adds the discharge of its own moulins at t_model + dt
// (the time the residual is forced at) before the reduction.
static void diagnostics_record(shakti_model* m, double dt, int its, double residual, double* row) {
  ensure_rules(m);
  const bool multi = comm().active(), moulins = m->n_moulins > 0;
  launch_diagnostics(m->hm.ne, m->c0.p, m->c1.p, m->c2.p, m->cell_counted.p, m->fields(), m->kbar.p, dt, m->dprm,
                     m->diag_parts, m->diag_partial.p, m->diag_vals.p, multi || moulins ? nullptr : row, its, residual,
                     m->stream);
  if (moulins) launch_diagnostics_moulins(m->diag_vals.p, owned_moulin_discharge(m, m->t_model + dt), m->stream);
  if (multi) {
    comm_allreduce_sum(m->diag_vals.p, kDiagSums, m->stream);
    comm_allreduce_max(m->diag_vals.p + kDiagSums, kDiagVals - kDiagSums, m->stream);
  }
  if (multi || moulins) launch_diagnostics_row(m->diag_vals.p, row, dt, its, residual, m->stream);
}

static void require_diag_rows(shakti_model* m, int64_t n) {
  if (m->diag_cap > 0 && n > m->diag_cap - m->diag_n)
    throw Error(SHAKTI_ERR_INVALID, "diagnostics buffer full (" + std::to_string(m->diag_n) + " of " +
                                        std::to_string(m->diag_cap) + " rows): read it with shakti_read_diagnostics");
}

static void newton_solve(shakti_model* m, double dt, int32_t* niter, int32_t* converged) {
  const int32_t no = m->hm.n_owned;
  static const bool trace = getenv("SHAKTI_TRACE_NEWTON") != nullptr;
  require_diag_rows(m, 1);
  compute_kbar(m);
  assemble(m, dt, 1);
  double r = norm2(m, m->F.p);
  const double r_init = r;
  auto rel_of = [&](double res) {
    if (m->opt.newton_r0 == SHAKTI_R0_DOLFINX) return m->residual0 > 0 ? res / m->residual0 : (double)INFINITY;
    return r_init > 0 ? res / r_init : 0.0;
  };
  auto check = [&](double res) { return rel_of(res) < m->opt.newton_rtol || res < m->opt.newton_atol; };
  // absolute residual below which the Newton test passes (unknown before the first dx in DOLFINx mode)
  auto newton_target = [&]() {
    const double den = m->opt.newton_r0 == SHAKTI_R0_DOLFINX ? m->residual0 : r_init;
    return std::max(m->opt.newton_atol, den > 0 ? m->opt.newton_rtol * den : 0.0);
  };
  bool conv = check(r);
  int it = 0;
  double r_prev = -1.0;
  // With the DOLFINx r0 the Newton test is loose and scale dependent (the iteration often stops long
  // before it has converged), so the iterate it stops at depends on every solve: no forcing there.
  // Likewise with an under-relaxed step the iteration converges linearly and the quadratic model behind
  // the forcing terms does not hold.
  const double relax = m->opt.newton_relaxation;
  SHAKTI_REQUIRE(relax > 0, "newton_relaxation must be positive");
  const double forcing = (m->opt.newton_r0 == SHAKTI_R0_DOLFINX || relax != 1.0) ? 0.0 : m->opt.linear_forcing;
  const bool hist_ok = m->hist_ratio > 0 && m->hist_dt > 0 && std::fabs(dt / m->hist_dt - 1.0) < 0.5;
  const double tau_tight = m->opt.linear_rtol * r_init;
  double tau_last = tau_tight;
  if (trace && comm().rank == 0) fprintf(stderr, "[newton] dt %.4g r0 %.6e\n", dt, r);
  while (!conv && it < m->opt.newton_max_it) {
    // Dirichlet rows are identity rows and their columns are zero: solve the interior system
    launch_xmy_masked(no, m->F.p, m->isbc.p, m->rhs.p, m->stream);
    m->newton_it_in_step = it;
    double tau = tau_tight, pred = -1.0;
    if (forcing > 0) {
      // only in the fast (quadratic) phase: while the residual falls by less than 10x per iteration the
      // solves stay tight and the iterates are those of the exact iteration
      if (it == 0) { if (hist_ok && m->hist_ratio < 0.1) pred = m->hist_ratio * r; }
      else if (r_prev > 0 && r < 0.1 * r_prev) pred = r * (r / r_prev) * (r / r_prev);
      if (pred >= 10.0 * newton_target()) tau = std::max(tau, forcing * pred);
    }
    tau_last = tau;
    const double rtol_k = std::min(1e-2, r > 0 ? tau / r : 1e-2);
    KrylovResult kr = linear_solve(m, m->rhs.p, m->dx.p, rtol_k);
    if (!kr.converged)
      throw Error(SHAKTI_ERR_LINEAR, "Krylov solve did not reach its tolerance (relres " +
                                         std::to_string(kr.relres) + " after " + std::to_string(kr.iterations) + " its)");
    if (m->n_bc) SHAKTI_LAUNCH(fix_bc_dx_kernel, div_up(no, 256), 256, 0, m->stream, no, m->isbc.p, m->F.p, m->dx.p);
    double lam = relax;
    launch_axpy(no, -lam, m->dx.p, m->N.p, m->stream);   // x <- x - relaxation dx   (relaxation = 1 in the reference)
    m->halo.exchange(m->N.p, m->stream);
    ++it;
    if (it == 1 && m->opt.newton_r0 == SHAKTI_R0_DOLFINX) m->residual0 = norm2(m, m->dx.p);
    // The Jacobian is only needed if another iteration follows: when the model says this one converged
    // with a decade to spare, assemble the residual alone (and the Jacobian after all if it did not)
    const bool expect_conv = forcing > 0 && pred >= 0 && 10.0 * (pred + tau) < newton_target();
    bool have_J = !expect_conv;
    assemble(m, dt, have_J ? 1 : 0);
    r_prev = r;
    r = norm2(m, m->F.p);
    // Backtracking line search (newton_line_search > 0; not in the reference): halve the step until the
    // residual norm has decreased sufficiently.  N currently holds x - lam dx; x - lam/2 dx = N + lam/2 dx.
    // A NaN residual (state outside the model's range) fails the test and is backtracked like an increase.
    int nb = 0;
    while (nb < m->opt.newton_line_search && !(r <= (1.0 - 1e-4 * lam) * r_prev)) {
      launch_axpy(no, 0.5 * lam, m->dx.p, m->N.p, m->stream);
      m->halo.exchange(m->N.p, m->stream);
      lam *= 0.5;
      ++nb;
      assemble(m, dt, 0);
      have_J = false;
      r = norm2(m, m->F.p);
    }
    m->st.newton_backtracks += nb;
    conv = check(r);
    if (!conv && !have_J) assemble(m, dt, 1);
    if (trace && comm().rank == 0)
      fprintf(stderr, "[newton]   it %d krylov %d (rtol %.2e) r %.6e rel %.3e step %.4g%s\n", it, kr.iterations, rtol_k, r,
              rel_of(r), lam, expect_conv ? " F-only" : "");
    if (it == 1) { m->hist_ratio = r_prev > 0 ? r / r_prev : -1.0; m->hist_dt = dt; }
    if (conv && tau_last > tau_tight) {
      // The iteration converged one step earlier than the model expected, i.e. after a LOOSE solve.  The
      // iterate must not depend on that: one more correction with the current Jacobian, solved tightly
      // (not counted as a Newton iteration -- the exact iteration would have stopped here too).
      if (!have_J) assemble(m, dt, 1);   // only after a backtracked step: the trial residuals were F-only
      launch_xmy_masked(no, m->F.p, m->isbc.p, m->rhs.p, m->stream);
      m->newton_it_in_step = it;
      KrylovResult kp = linear_solve(m, m->rhs.p, m->dx.p, std::min(1e-2, r > 0 ? tau_tight / r : 1e-2));
      if (kp.converged) {
        if (m->n_bc) SHAKTI_LAUNCH(fix_bc_dx_kernel, div_up(no, 256), 256, 0, m->stream, no, m->isbc.p, m->F.p, m->dx.p);
        launch_axpy(no, -1.0, m->dx.p, m->N.p, m->stream);
        m->halo.exchange(m->N.p, m->stream);
        assemble(m, dt, 0);
        r = norm2(m, m->F.p);
        if (trace && comm().rank == 0) fprintf(stderr, "[newton]   polish krylov %d r %.6e\n", kp.iterations, r);
      }
    }
  }
  if (it == 0) m->hist_ratio = -1.0;
  m->st.newton_its += it;
  m->st.last_residual = r;
  m->st.last_residual0 = m->opt.newton_r0 == SHAKTI_R0_DOLFINX ? m->residual0 : r_init;
  *niter = it;
  *converged = conv ? 1 : 0;
  if (!conv) throw Error(SHAKTI_ERR_NOT_CONVERGED, "Newton solver did not converge");
  if (m->diag_cap > 0) {   // Kbar and h0 are those of the solve
    diagnostics_record(m, dt, it, r, m->diag_rows.p + m->diag_n * SHAKTI_D_COUNT);
    m->diag_n++;
  }
}

static void update_q(shakti_model* m) {
  refresh_h0(m);
  launch_update_q(m->hm.n_owned, m->win.p, m->x.p, m->y.p, m->h0.p, m->N.p, m->b.p, m->qx.p, m->qy.p, m->dprm, m->stream);
}
static void update_melt(shakti_model* m) {
  refresh_h0(m);
  launch_update_melt(m->hm.n_owned, m->win.p, m->x.p, m->y.p, m->h0.p, m->N.p, m->b.p, m->qx.p, m->qy.p, m->G.p,
                     m->melt.p, m->melt2.p, m->dprm, m->stream);
  std::swap(m->melt.p, m->melt2.p);
  m->halo.exchange(m->melt.p, m->stream);
}
// q and melt_n in one pass (what shakti_step uses; identical results to update_q + update_melt)
static void update_q_melt(shakti_model* m) {
  SHAKTI_PHASE("nodal_q_melt", m->stream);
  refresh_h0(m);
  launch_update_q_melt(m->hm.n_owned, m->win.p, m->x.p, m->y.p, m->h0.p, m->N.p, m->b.p, m->qx.p, m->qy.p, m->G.p,
                       m->melt.p, m->melt2.p, m->dprm, m->stream);
  std::swap(m->melt.p, m->melt2.p);
  m->halo.exchange(m->melt.p, m->stream);
}
static void update_b(shakti_model* m, double dt) {
  SHAKTI_PHASE("nodal_b", m->stream);
  refresh_h0(m);
  launch_update_b(m->hm.n_owned, m->win.p, m->x.p, m->y.p, m->h0.p, m->N.p, m->b.p, m->qx.p, m->qy.p, m->G.p,
                  m->melt.p, m->b2.p, dt, m->opt.b_min, m->dprm, m->stream);
  std::swap(m->b.p, m->b2.p);
  m->halo.exchange(m->b.p, m->stream);
  m->halo.exchange(m->qx.p, m->stream);
  m->halo.exchange(m->qy.p, m->stream);
  // the gap-height update closes a time step on both paths (shakti_step and the split entry points
  // solvers.solve(md) drives), so the step counter -- and with it amg_refresh_every -- advances here, and so does
  // the model clock
  m->st.steps++;
  m->t_model += dt;
}
static void copy_N(shakti_model* m) {
  SHAKTI_CUDA(cudaMemcpyAsync(m->N_n.p, m->N.p, sizeof(double) * m->hm.n_local, cudaMemcpyDeviceToDevice, m->stream));
}

static void step(shakti_model* m, double dt, int32_t* niter, int32_t* converged) {
  SHAKTI_REQUIRE(dt > 0, "dt must be positive");
  int32_t it = 0, cv = 0;
  {
    SHAKTI_PHASE("step_total", m->stream);
    newton_solve(m, dt, &it, &cv);
    update_q_melt(m);
    update_b(m, dt);
    copy_N(m);
  }
  if (phase_trace_enabled() && comm().rank == 0) phase_report("step");
  if (niter) *niter = it;
  if (converged) *converged = cv;
}

// Snapshot b, N, qx, qy on the compute stream and enqueue their device->host copies on the copy stream
// (see shakti_step_host_async in the header).
static void save_outputs_async(shakti_model* m, double* b_out, double* N_out, double* qx_out, double* qy_out, int owned_only) {
  const HostMesh& hm = m->hm;
  const size_t n_out = owned_only ? (size_t)hm.n_owned : (size_t)hm.nv_g;
  double* outs[4] = {b_out, N_out, qx_out, qy_out};
  const double* src[4] = {m->b.p, m->N.p, m->qx.p, m->qy.p};
  bool any = false;
  for (int k = 0; k < 4; ++k) any |= outs[k] != nullptr;
  if (!any) return;
  // the previous snapshots must have left the device before they are overwritten (a D2H of the
  // previous save is far shorter than a step, so this wait is free in practice)
  if (m->d2h_pending) SHAKTI_CUDA(cudaStreamWaitEvent(m->stream, m->ev_d2h, 0));
  for (int k = 0; k < 4; ++k) {
    if (!outs[k]) continue;
    if (m->out_stage[k].n < n_out) m->out_stage[k].alloc(std::max<size_t>(n_out, 1));
    if (owned_only) {
      if (n_out) SHAKTI_CUDA(cudaMemcpyAsync(m->out_stage[k].p, src[k], sizeof(double) * n_out, cudaMemcpyDeviceToDevice, m->stream));
    } else {
      gather_out(m, src[k], m->out_stage[k].p);
    }
  }
  SHAKTI_CUDA(cudaEventRecord(m->ev_snap, m->stream));
  SHAKTI_CUDA(cudaStreamWaitEvent(m->copy_stream, m->ev_snap, 0));
  // in chunks: the copy engine serves its queue in order, and a step's small reads (when they go through it)
  // must not wait behind a whole 128 MB field
  const char* ce = getenv("SHAKTI_D2H_CHUNK_MB");
  const size_t chunk = (size_t)(ce ? std::max(1, atoi(ce)) : 8) << 17;   // doubles per chunk (MB * 2^20 / 8)
  for (int k = 0; k < 4; ++k)
    if (outs[k] && n_out)
      for (size_t o = 0; o < n_out; o += chunk)
        SHAKTI_CUDA(cudaMemcpyAsync(outs[k] + o, m->out_stage[k].p + o, sizeof(double) * std::min(chunk, n_out - o),
                                    cudaMemcpyDeviceToHost, m->copy_stream));
  SHAKTI_CUDA(cudaEventRecord(m->ev_d2h, m->copy_stream));
  m->d2h_pending = true;
}

static bool is_dirichlet(const shakti_model* m, int32_t v) { return std::binary_search(m->bc_g.begin(), m->bc_g.end(), v); }

static void set_dirichlet(shakti_model* m, const int32_t* dofs, int64_t n, double value) {
  std::vector<uint8_t> flag(m->hm.n_local, 0);
  for (int64_t i = 0; i < n; ++i) {
    SHAKTI_REQUIRE(dofs[i] >= 0 && dofs[i] < m->hm.nv_g, "Dirichlet dof out of range");
    const int32_t l = m->hm.g2l[dofs[i]];
    if (l >= 0) flag[l] = 1;
  }
  std::vector<int32_t> bc(dofs, dofs + n);
  std::sort(bc.begin(), bc.end());
  for (int64_t k = 0; k < m->n_moulins; ++k)
    if (std::binary_search(bc.begin(), bc.end(), m->mo_vertex[k]))
      throw Error(SHAKTI_ERR_INVALID, "Dirichlet dof " + std::to_string(m->mo_vertex[k]) + " carries moulin " +
                                          std::to_string(k) + ": remove or move the moulin first");
  m->bc_g.swap(bc);
  m->isbc.upload(flag);
  m->N_bdry = value;
  m->n_bc = n;   // global count: >0 on every rank
  m->hist_ratio = -1.0;
  m->amg_setup_done = false;  // excluded rows changed
  m->amg.reset();
}

// Validate everything before any state changes; then keep the hydrographs on the host and upload this rank's
// moulin rows (owned vertices only: ghosts belong to another rank) sorted by row, caller order within a row.
static void set_moulins(shakti_model* m, int64_t n, const int32_t* vertex, const int64_t* knot_ptr, const double* t_knots,
                        const double* q_knots, double period) {
  SHAKTI_REQUIRE(n >= 0 && n < ((int64_t)1 << 31), "n_moulins out of range");
  SHAKTI_REQUIRE(std::isfinite(period) && period >= 0, "moulin period must be finite and >= 0 (0: no period)");
  if (n > 0) SHAKTI_REQUIRE(vertex && knot_ptr && t_knots && q_knots, "null moulin argument");
  if (n > 0) SHAKTI_REQUIRE(knot_ptr[0] == 0, "knot_ptr[0] must be 0");
  for (int64_t k = 0; k < n; ++k) {
    const std::string who = "moulin " + std::to_string(k);
    SHAKTI_REQUIRE(vertex[k] >= 0 && vertex[k] < m->hm.nv_g, who + ": vertex out of range");
    if (is_dirichlet(m, vertex[k]))
      throw Error(SHAKTI_ERR_INVALID, who + ": vertex " + std::to_string(vertex[k]) + " is a Dirichlet dof");
    SHAKTI_REQUIRE(knot_ptr[k + 1] > knot_ptr[k], who + ": empty hydrograph");
    for (int64_t j = knot_ptr[k]; j < knot_ptr[k + 1]; ++j) {
      SHAKTI_REQUIRE(std::isfinite(t_knots[j]) && std::isfinite(q_knots[j]), who + ": knot times and discharges must be finite");
      SHAKTI_REQUIRE(j == knot_ptr[k] || t_knots[j] > t_knots[j - 1], who + ": knot times must be strictly increasing");
    }
  }
  const int64_t nk = n > 0 ? knot_ptr[n] : 0;
  std::vector<int64_t> own;
  for (int64_t k = 0; k < n; ++k) {
    const int32_t l = m->hm.g2l[vertex[k]];
    if (l >= 0 && l < m->hm.n_owned) own.push_back(k);
  }
  std::stable_sort(own.begin(), own.end(), [&](int64_t a, int64_t b) { return m->hm.g2l[vertex[a]] < m->hm.g2l[vertex[b]]; });
  std::vector<int32_t> row, rptr;
  std::vector<int64_t> kptr(1, 0);
  std::vector<double> tk, qk;
  for (size_t i = 0; i < own.size(); ++i) {
    const int64_t k = own[i];
    const int32_t l = m->hm.g2l[vertex[k]];
    if (row.empty() || row.back() != l) { row.push_back(l); rptr.push_back((int32_t)i); }
    tk.insert(tk.end(), t_knots + knot_ptr[k], t_knots + knot_ptr[k + 1]);
    qk.insert(qk.end(), q_knots + knot_ptr[k], q_knots + knot_ptr[k + 1]);
    kptr.push_back((int64_t)tk.size());
  }
  rptr.push_back((int32_t)own.size());
  SHAKTI_CUDA(cudaStreamSynchronize(m->stream));   // a queued assembly may still read the old tables
  m->mo_row_d.upload(row);
  m->mo_rptr_d.upload(rptr);
  m->mo_kptr_d.upload(kptr);
  m->mo_t_d.upload(tk);
  m->mo_q_d.upload(qk);
  m->mo_rows = (int32_t)row.size();
  m->n_moulins = n;
  m->mo_vertex.assign(vertex, vertex + n);
  m->mo_kptr.assign(knot_ptr, knot_ptr + n + (n > 0));
  m->mo_t.assign(t_knots, t_knots + nk);
  m->mo_q.assign(q_knots, q_knots + nk);
  m->mo_period = period;
  m->mo_own.swap(own);
}

static HostCsr& caller_pattern(shakti_model* m) {
  if (!m->csr_g) m->csr_g.reset(new HostCsr(caller_csr(m->hm.nv_g, m->hm.ne_g, m->cells_g.data())));
  return *m->csr_g;
}

static void create(int64_t nv, int64_t ne, const double* xy, const int32_t* cells, const shakti_params* params,
                   const shakti_options* opt, int device, shakti_model** out) {
  SHAKTI_REQUIRE(out && xy && cells, "null argument");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    throw Error(SHAKTI_ERR_NO_DEVICE, "no CUDA device: the SHAKTI B200 path has no CPU fallback");
  }
  std::unique_ptr<shakti_model> m(new shakti_model());
  if (device < 0) SHAKTI_CUDA(cudaGetDevice(&device));
  m->device = device;
  SHAKTI_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  SHAKTI_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10)
    throw Error(SHAKTI_ERR_NO_DEVICE, std::string("device '") + prop.name + "' is not sm_100 class; this library is built for sm_100a only");
  m->sm_count = prop.multiProcessorCount;
  SHAKTI_CUDA(cudaStreamCreateWithFlags(&m->stream, cudaStreamNonBlocking));
  SHAKTI_CUDA(cudaStreamCreateWithFlags(&m->copy_stream, cudaStreamNonBlocking));
  SHAKTI_CUDA(cudaEventCreateWithFlags(&m->ev_snap, cudaEventDisableTiming));
  SHAKTI_CUDA(cudaEventCreateWithFlags(&m->ev_d2h, cudaEventDisableTiming));
  if (params) m->prm = *params; else shakti_default_params(&m->prm);
  if (opt) m->opt = *opt; else shakti_default_options(&m->opt);
  m->dprm = make_dev_params(m->prm);
  m->launches_at_create = g_kernel_launches;
  m->cells_g.assign(cells, cells + 3 * ne);
  build_host_mesh(nv, ne, xy, cells, comm().rank, comm().nranks, m->opt.reorder, m->hm);
  HostMesh& hm = m->hm;
  // device mesh
  m->x.upload(hm.x);
  m->y.upload(hm.y);
  {
    std::vector<int32_t> a(hm.ne), b(hm.ne), c(hm.ne);
    for (int32_t e = 0; e < hm.ne; ++e) { a[e] = hm.cells[3 * (size_t)e]; b[e] = hm.cells[3 * (size_t)e + 1]; c[e] = hm.cells[3 * (size_t)e + 2]; }
    m->c0.upload(a); m->c1.upload(b); m->c2.upload(c);
  }
  m->slot.upload(hm.slot);
  {
    const char* env = getenv("SHAKTI_ASM_MAX_CELLS");   // tuning knob: smaller => fewer rows per block
    // <= 400 cells per block => 128-row blocks of 128 threads, ~48 KB of shared memory, 4 blocks/SM
    // (measured at 16M dofs: 3.02 ms vs 3.24 ms with 256-row blocks)
    build_assembly_blocks(hm, env ? atoi(env) : 400, m->ab);
  }      // <= 800 cells per block: 77 KB of staged cell data + ~35 KB of vertex data
  if (m->ab.ok) {
    m->ab_eptr.upload(m->ab.blk_eptr);
    m->ab_elems.upload(m->ab.blk_elems);
    m->ab_incptr.upload(m->ab.inc_ptr);
    m->ab_inc.upload(m->ab.inc_code);
    m->ab_src.upload(m->ab.src);
    m->ab_lv.upload(m->ab.blk_lv);
    m->ab_hptr.upload(m->ab.blk_hptr);
    m->ab_halo.upload(m->ab.blk_halo);
    std::vector<uint16_t>().swap(m->ab.blk_lv);
    std::vector<int32_t>().swap(m->ab.blk_halo);
    // host copies are only needed for the plan itself
    std::vector<int32_t>().swap(m->ab.blk_elems);
    std::vector<uint16_t>().swap(m->ab.inc_code);
    std::vector<uint32_t>().swap(m->ab.src);
  }
  m->diag_pos.upload(hm.diag_pos);
  m->cell_counted.upload(std::vector<uint8_t>(hm.cell_counted.begin(), hm.cell_counted.end()));
  m->diag_parts = diagnostics_parts(hm.ne, m->sm_count);
  m->diag_partial.alloc((size_t)m->diag_parts * kDiagVals);
  m->diag_vals.alloc(kDiagVals + SHAKTI_D_COUNT);
  m->win.upload(hm.win);
  m->l2g.upload(hm.l2g);
  const size_t nl = std::max<int32_t>(hm.n_local, 1);
  for (DevBuf<double>* f : {&m->z_b, &m->z_s, &m->h0, &m->G, &m->inputs, &m->storage, &m->b, &m->b2, &m->N, &m->N_n,
                            &m->qx, &m->qy, &m->melt, &m->melt2, &m->F, &m->dx, &m->rhs, &m->dinv})
    f->alloc_zero(nl, m->stream);
  m->kbar.alloc_zero(std::max<int32_t>(hm.ne, 1), m->stream);
  m->isbc.alloc_zero(nl, m->stream);
  m->stage.alloc((size_t)nv);
  m->scal.alloc_zero(16, m->stream);
  SHAKTI_CUDA(cudaMallocHost(&m->host_scal, 16 * sizeof(double)));
  m->J.upload_pattern(hm.S, hm.A.nnz());
  m->halo.build(hm.nbrs);
  m->red.init(m->sm_count);
  m->gmres.init(hm.n_owned, hm.n_local, std::max(2, m->opt.gmres_restart), m->sm_count, m->stream);
  // quadrature tables
  default_k_rule(m->kq_pts, m->kq_wts);
  g_rule_owner = nullptr;
  ensure_rules(m.get());
  // stats
  m->st.n_vert = nv; m->st.n_cell = ne;
  m->st.n_owned = hm.n_owned; m->st.n_local = hm.n_local; m->st.n_cell_local = hm.ne; m->st.nnz_local = hm.A.nnz();
  m->st.nnz = comm().active() ? -1 : hm.A.nnz();
  SHAKTI_CUDA(cudaStreamSynchronize(m->stream));
  *out = m.release();
}

static void destroy(shakti_model* m) {
  if (!m) return;
  if (g_rule_owner == m) g_rule_owner = nullptr;
  cudaSetDevice(m->device);
  if (m->stream) cudaStreamSynchronize(m->stream);
  // swap-safe: DevBuf destructors free whatever pointer they currently hold
  if (m->host_scal) cudaFreeHost(m->host_scal);
  if (m->copy_stream) { cudaStreamSynchronize(m->copy_stream); cudaStreamDestroy(m->copy_stream); }
  if (m->ev_snap) cudaEventDestroy(m->ev_snap);
  if (m->ev_d2h) cudaEventDestroy(m->ev_d2h);
  cudaStream_t s = m->stream;
  delete m;
  if (s) cudaStreamDestroy(s);
}

// n-point Gauss rule for the weight (1-x)^alpha (1+x)^beta on [-1,1] by Golub-Welsch: nodes are
// the eigenvalues of the Jacobi matrix of the monic recurrence, weights mu0 * (first eigenvector
// component)^2.  The small symmetric eigenproblem is solved with cyclic Jacobi rotations.
static void gauss_jacobi(int n, long double alpha, long double beta, std::vector<long double>& x,
                         std::vector<long double>& w) {
  std::vector<long double> T((size_t)n * n, 0.0L), Q((size_t)n * n, 0.0L);
  const long double ab = alpha + beta;
  for (int k = 0; k < n; ++k) {
    long double a;
    if (k == 0) a = (beta - alpha) / (ab + 2.0L);
    else a = (beta * beta - alpha * alpha) / ((2.0L * k + ab) * (2.0L * k + ab + 2.0L));
    T[(size_t)k * n + k] = a;
    if (k >= 1) {
      long double b;
      if (k == 1) b = 4.0L * (1.0L + alpha) * (1.0L + beta) / ((2.0L + ab) * (2.0L + ab) * (3.0L + ab));
      else {
        const long double t = 2.0L * k + ab;
        b = 4.0L * k * (k + alpha) * (k + beta) * (k + ab) / (t * t * (t + 1.0L) * (t - 1.0L));
      }
      T[(size_t)k * n + k - 1] = T[(size_t)(k - 1) * n + k] = std::sqrt(b);
    }
    Q[(size_t)k * n + k] = 1.0L;
  }
  for (int sweep = 0; sweep < 100; ++sweep) {
    long double off = 0.0L;
    for (int p = 0; p < n; ++p)
      for (int q = p + 1; q < n; ++q) off += T[(size_t)p * n + q] * T[(size_t)p * n + q];
    if (off < 1e-40L) break;
    for (int p = 0; p < n; ++p)
      for (int q = p + 1; q < n; ++q) {
        const long double apq = T[(size_t)p * n + q];
        if (apq == 0.0L) continue;
        const long double theta = (T[(size_t)q * n + q] - T[(size_t)p * n + p]) / (2.0L * apq);
        const long double t = (theta >= 0 ? 1.0L : -1.0L) / (std::fabs(theta) + std::sqrt(theta * theta + 1.0L));
        const long double c = 1.0L / std::sqrt(t * t + 1.0L), sn = t * c;
        for (int k = 0; k < n; ++k) {  // columns p,q of T
          const long double kp = T[(size_t)k * n + p], kq = T[(size_t)k * n + q];
          T[(size_t)k * n + p] = c * kp - sn * kq;
          T[(size_t)k * n + q] = sn * kp + c * kq;
        }
        for (int k = 0; k < n; ++k) {  // rows p,q of T
          const long double pk = T[(size_t)p * n + k], qk = T[(size_t)q * n + k];
          T[(size_t)p * n + k] = c * pk - sn * qk;
          T[(size_t)q * n + k] = sn * pk + c * qk;
        }
        for (int k = 0; k < n; ++k) {  // accumulate eigenvectors (columns of Q)
          const long double kp = Q[(size_t)k * n + p], kq = Q[(size_t)k * n + q];
          Q[(size_t)k * n + p] = c * kp - sn * kq;
          Q[(size_t)k * n + q] = sn * kp + c * kq;
        }
      }
  }
  const long double mu0 = std::pow(2.0L, ab + 1.0L) * std::tgamma(alpha + 1.0L) * std::tgamma(beta + 1.0L) /
                          std::tgamma(ab + 2.0L);
  std::vector<int> order(n);
  for (int i = 0; i < n; ++i) order[i] = i;
  std::sort(order.begin(), order.end(), [&](int a, int b) { return T[(size_t)a * n + a] < T[(size_t)b * n + b]; });
  x.resize(n);
  w.resize(n);
  for (int i = 0; i < n; ++i) {
    const int j = order[i];
    x[i] = T[(size_t)j * n + j];
    w[i] = mu0 * Q[j] * Q[j];  // first row of Q, column j
  }
}

// collapsed (Duffy) Gauss-Jacobi rule of degree 7: 4 x 4 points, weights sum to 1/2
static void default_k_rule(std::vector<double>& pts, std::vector<double>& wts) {
  std::vector<long double> xu, wu, xv, wv;
  gauss_jacobi(4, 1.0L, 0.0L, xu, wu);
  gauss_jacobi(4, 0.0L, 0.0L, xv, wv);
  pts.clear();
  wts.clear();
  for (int i = 0; i < 4; ++i)
    for (int j = 0; j < 4; ++j) {
      const long double u = 0.5L * (1.0L + xu[i]), v = 0.5L * (1.0L + xv[j]);
      pts.push_back((double)u);
      pts.push_back((double)(v * (1.0L - u)));
      wts.push_back((double)(0.25L * wu[i] * 0.5L * wv[j]));
    }
}

}  // namespace shakti

// ====================================================================== extern "C"
#define SHAKTI_TRY try {
#define SHAKTI_CATCH                                      \
  }                                                       \
  catch (const shakti::Error& e) {                        \
    shakti::set_last_error(e.what());                     \
    return e.code;                                        \
  }                                                       \
  catch (const std::exception& e) {                       \
    shakti::set_last_error(e.what());                     \
    return SHAKTI_ERR_INVALID;                            \
  }                                                       \
  return SHAKTI_OK;

extern "C" {

const char* shakti_last_error(void) { return shakti::t_last_error.c_str(); }
const char* shakti_version(void) { return "shakti_b200 0.1 (sm_100a)"; }

int shakti_device_count(int* n) {
  if (!n) return SHAKTI_ERR_INVALID;
  *n = 0;
  if (cudaGetDeviceCount(n) != cudaSuccess) { cudaGetLastError(); *n = 0; }
  return SHAKTI_OK;
}

int shakti_default_params(shakti_params* p) {
  if (!p) return SHAKTI_ERR_INVALID;
  p->g = 9.81; p->rho_i = 917; p->rho_w = 1000; p->nu = 1.787e-6; p->Lh = 3.34e5; p->omega = 1e-3; p->n = 3; p->A = 2.24e-24;
  return SHAKTI_OK;
}

int shakti_default_options(shakti_options* o) {
  if (!o) return SHAKTI_ERR_INVALID;
  o->newton_rtol = 1e-9; o->newton_atol = 1e-10; o->newton_max_it = 50; o->newton_r0 = SHAKTI_R0_INITIAL_RESIDUAL;
  o->linear_solver = SHAKTI_KSP_GMRES; o->precond = SHAKTI_PC_AMG;
  o->linear_rtol = 1e-12; o->linear_atol = 0.0; o->linear_max_it = 2000; o->gmres_restart = 40;
  o->amg_refresh_every = 2; o->amg_max_levels = 12; o->amg_coarse_size = 256; o->amg_presmooth = 2; o->amg_postsmooth = 2;
  o->amg_smoother_omega = 0.67; o->amg_prolong_omega = 0.67; o->amg_strength_theta = 0.08; o->amg_cheby_ratio = 5.0;
  o->amg_smoother = 1; o->amg_fp32_cycle = 1; o->amg_cuda_graph = 1; o->amg_smoother_halo = 1;
  o->b_min = 1.0e-5; o->assembly_kernel = 0; o->reorder = 1;
  o->linear_forcing = 0.01;
  o->amg_replicate_below = 100000;
  o->newton_relaxation = 1.0;
  o->newton_line_search = 0;
  return SHAKTI_OK;
}

int shakti_create(int64_t n_vert, int64_t n_cell, const double* xy, const int32_t* cells, const shakti_params* params,
                  const shakti_options* opt, int device, shakti_model** out) {
  SHAKTI_TRY
  shakti::create(n_vert, n_cell, xy, cells, params, opt, device, out);
  SHAKTI_CATCH
}

int shakti_destroy(shakti_model* m) {
  SHAKTI_TRY
  shakti::destroy(m);
  SHAKTI_CATCH
}

int shakti_set_field(shakti_model* m, int field, const double* src, int is_device) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(m, "null model");
  use_device(m);
  shakti::set_field(m, field, src, is_device);
  SHAKTI_CATCH
}
int shakti_get_field(shakti_model* m, int field, double* dst, int is_device) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(m, "null model");
  use_device(m);
  shakti::get_field(m, field, dst, is_device);
  SHAKTI_CATCH
}

int shakti_set_flux(shakti_model* m, const double* q, int is_device) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(m && q, "null argument");
  use_device(m);
  m->hist_ratio = -1.0;
  const int64_t nv = m->hm.nv_g;
  if (!m->stage2.p) m->stage2.alloc((size_t)3 * nv);
  const double* src = q;
  if (!is_device) {
    SHAKTI_CUDA(cudaMemcpyAsync(m->stage2.p, q, sizeof(double) * 2 * nv, cudaMemcpyHostToDevice, m->stream));
    src = m->stage2.p;
  }
  double* tmp = m->stage2.p + 2 * nv;
  launch_deinterleave(nv, src, m->stage.p, tmp, m->stream);
  scatter_in(m, m->stage.p, m->qx.p);
  scatter_in(m, tmp, m->qy.p);
  SHAKTI_CUDA(cudaStreamSynchronize(m->stream));
  SHAKTI_CATCH
}
int shakti_get_flux(shakti_model* m, double* q, int is_device) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(m && q, "null argument");
  use_device(m);
  const int64_t nv = m->hm.nv_g;
  if (!m->stage2.p) m->stage2.alloc((size_t)3 * nv);
  double* tmp = m->stage2.p + 2 * nv;
  gather_out(m, m->qx.p, m->stage.p);
  gather_out(m, m->qy.p, tmp);
  double* dst = is_device ? q : m->stage2.p;
  launch_interleave(nv, m->stage.p, tmp, dst, m->stream);
  if (!is_device) SHAKTI_CUDA(cudaMemcpyAsync(q, dst, sizeof(double) * 2 * nv, cudaMemcpyDeviceToHost, m->stream));
  SHAKTI_CUDA(cudaStreamSynchronize(m->stream));
  SHAKTI_CATCH
}

int shakti_set_dirichlet(shakti_model* m, const int32_t* dofs, int64_t n_dofs, double value) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(m && (dofs || n_dofs == 0) && n_dofs >= 0, "bad Dirichlet arguments");
  use_device(m);
  shakti::set_dirichlet(m, dofs, n_dofs, value);
  SHAKTI_CATCH
}

int shakti_locate_dirichlet(shakti_model* m, const uint8_t* marker, int32_t* dofs, int64_t cap, int64_t* n_out) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(m && marker && n_out, "null argument");
  std::vector<int32_t> d = locate_dirichlet_dofs(m->hm.nv_g, m->hm.ne_g, m->cells_g.data(), marker);
  *n_out = (int64_t)d.size();
  if (dofs) {
    SHAKTI_REQUIRE(cap >= (int64_t)d.size(), "dof buffer too small");
    std::copy(d.begin(), d.end(), dofs);
  }
  SHAKTI_CATCH
}

int shakti_set_quadrature(shakti_model* m, int32_t n_pts, const double* pts_xy, const double* wts) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(m && pts_xy && wts && n_pts > 0 && n_pts <= 64, "quadrature table must have 1..64 points");
  use_device(m);
  m->kq_pts.assign(pts_xy, pts_xy + 2 * n_pts);
  m->kq_wts.assign(wts, wts + n_pts);
  g_rule_owner = nullptr;
  ensure_rules(m);
  SHAKTI_CATCH
}

int shakti_set_options(shakti_model* m, const shakti_options* opt) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(m && opt, "null argument");
  use_device(m);
  const bool amg_changed = opt->amg_max_levels != m->opt.amg_max_levels || opt->amg_coarse_size != m->opt.amg_coarse_size ||
                           opt->amg_presmooth != m->opt.amg_presmooth || opt->amg_postsmooth != m->opt.amg_postsmooth ||
                           opt->amg_smoother_omega != m->opt.amg_smoother_omega ||
                           opt->amg_prolong_omega != m->opt.amg_prolong_omega ||
                           opt->amg_strength_theta != m->opt.amg_strength_theta ||
                           opt->amg_cheby_ratio != m->opt.amg_cheby_ratio || opt->amg_smoother != m->opt.amg_smoother ||
                           opt->amg_fp32_cycle != m->opt.amg_fp32_cycle || opt->amg_cuda_graph != m->opt.amg_cuda_graph ||
                           opt->amg_smoother_halo != m->opt.amg_smoother_halo ||
                           opt->amg_replicate_below != m->opt.amg_replicate_below;
  SHAKTI_REQUIRE(opt->reorder == m->opt.reorder, "reorder can only be chosen at create time");
  const int restart_old = m->opt.gmres_restart;
  m->opt = *opt;
  m->hist_ratio = -1.0;
  if (amg_changed) { m->amg.reset(); m->amg_setup_done = false; }
  if (opt->gmres_restart != restart_old)
    m->gmres.init(m->hm.n_owned, m->hm.n_local, std::max(2, opt->gmres_restart), m->sm_count, m->stream);
  SHAKTI_CATCH
}
int shakti_get_options(shakti_model* m, shakti_options* opt) {
  if (!m || !opt) return SHAKTI_ERR_INVALID;
  *opt = m->opt;
  return SHAKTI_OK;
}
int shakti_get_stats(shakti_model* m, shakti_stats* st) {
  if (!m || !st) return SHAKTI_ERR_INVALID;
  m->st.kernel_launches = g_kernel_launches - m->launches_at_create;
  m->st.amg_levels = m->amg ? m->amg->levels() : 0;
  m->st.amg_operator_complexity = m->amg ? m->amg->operator_complexity() : 0.0;
  *st = m->st;
  return SHAKTI_OK;
}

int shakti_get_csr(shakti_model* m, int32_t* rowptr, int32_t* col, int64_t* nnz) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(m && nnz, "null argument");
  HostCsr& a = caller_pattern(m);
  *nnz = a.nnz();
  if (rowptr) std::copy(a.rowptr.begin(), a.rowptr.end(), rowptr);
  if (col) std::copy(a.col.begin(), a.col.end(), col);
  SHAKTI_CATCH
}

int shakti_kbar(shakti_model* m, double* out) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(m && out, "null argument");
  use_device(m);
  compute_kbar(m);
  std::vector<double> k = m->kbar.download(m->stream);
  for (int64_t e = 0; e < m->hm.ne_g; ++e) out[e] = 0.0;
  for (int32_t e = 0; e < m->hm.ne; ++e) out[m->hm.cell_l2g[e]] = k[e];
  SHAKTI_CATCH
}

int shakti_assemble(shakti_model* m, double dt, double* F_out, double* Jvals_out) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(m && dt > 0, "bad arguments");
  use_device(m);
  compute_kbar(m);
  assemble(m, dt, 1);
  if (F_out) shakti::get_field(m, SHAKTI_F_RESIDUAL, F_out, 0);
  if (Jvals_out) {
    HostCsr& a = caller_pattern(m);
    std::vector<double> v = m->J.val.download(m->stream);
    std::fill(Jvals_out, Jvals_out + a.nnz(), 0.0);
    const HostMesh& hm = m->hm;
    for (int32_t r = 0; r < hm.n_owned; ++r) {
      const int32_t gr = hm.l2g[r];
      const int32_t* b = a.col.data() + a.rowptr[gr];
      const int32_t* e = a.col.data() + a.rowptr[gr + 1];
      for (int32_t k = hm.A.rowptr[r]; k < hm.A.rowptr[r + 1]; ++k) {
        const int32_t gc = hm.l2g[hm.A.col[k]];
        const int32_t* p = std::lower_bound(b, e, gc);
        Jvals_out[p - a.col.data()] = v[hm.S.pos(r, k - hm.A.rowptr[r])];
      }
    }
  }
  SHAKTI_CATCH
}

int shakti_spmv(shakti_model* m, const double* x, double* y) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(m && x && y, "null argument");
  use_device(m);
  SHAKTI_REQUIRE(m->J_valid, "no assembled Jacobian");
  SHAKTI_CUDA(cudaMemcpyAsync(m->stage.p, x, sizeof(double) * m->hm.nv_g, cudaMemcpyHostToDevice, m->stream));
  scatter_in(m, m->stage.p, m->b2.p);   // b2 is scratch outside update_b
  launch_spmv(view(m->J), m->b2.p, m->rhs.p, m->stream);
  gather_out(m, m->rhs.p, m->stage.p);
  SHAKTI_CUDA(cudaMemcpyAsync(y, m->stage.p, sizeof(double) * m->hm.nv_g, cudaMemcpyDeviceToHost, m->stream));
  SHAKTI_CUDA(cudaStreamSynchronize(m->stream));
  SHAKTI_CATCH
}

int shakti_linear_solve(shakti_model* m, const double* rhs, double* dx, int32_t* iters, double* relres) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(m && rhs && dx, "null argument");
  use_device(m);
  SHAKTI_CUDA(cudaMemcpyAsync(m->stage.p, rhs, sizeof(double) * m->hm.nv_g, cudaMemcpyHostToDevice, m->stream));
  scatter_in(m, m->stage.p, m->b2.p);
  // interior system: Dirichlet rows are identity
  launch_xmy_masked(m->hm.n_owned, m->b2.p, m->isbc.p, m->rhs.p, m->stream);
  m->newton_it_in_step = 0;
  m->step_of_refresh = -1000000;   // parity hook: always refresh
  KrylovResult r = linear_solve(m, m->rhs.p, m->dx.p, m->opt.linear_rtol);
  if (m->n_bc)
    SHAKTI_LAUNCH(fix_bc_dx_kernel, div_up(m->hm.n_owned, 256), 256, 0, m->stream, m->hm.n_owned, m->isbc.p, m->b2.p, m->dx.p);
  gather_out(m, m->dx.p, m->stage.p);
  SHAKTI_CUDA(cudaMemcpyAsync(dx, m->stage.p, sizeof(double) * m->hm.nv_g, cudaMemcpyDeviceToHost, m->stream));
  SHAKTI_CUDA(cudaStreamSynchronize(m->stream));
  if (iters) *iters = r.iterations;
  if (relres) *relres = r.relres;
  if (!r.converged) throw Error(SHAKTI_ERR_LINEAR, "Krylov solve did not reach its tolerance");
  SHAKTI_CATCH
}

int shakti_get_winning_cells(shakti_model* m, int32_t* win_cell) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(m && win_cell, "null argument");
  for (int64_t i = 0; i < m->hm.nv_g; ++i) win_cell[i] = -1;
  for (int32_t r = 0; r < m->hm.n_owned; ++r) win_cell[m->hm.l2g[r]] = m->hm.win_cell[r];
  SHAKTI_CATCH
}

int shakti_start(shakti_model* m) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(m, "null model");
  use_device(m);
  SHAKTI_CUDA(cudaMemcpyAsync(m->N.p, m->N_n.p, sizeof(double) * m->hm.n_local, cudaMemcpyDeviceToDevice, m->stream));
  SHAKTI_CATCH
}

int shakti_newton_solve(shakti_model* m, double dt, int32_t* niter, int32_t* converged) {
  int32_t it = 0, cv = 0;
  if (niter) *niter = 0;
  if (converged) *converged = 0;
  SHAKTI_TRY
  SHAKTI_REQUIRE(m && dt > 0, "bad arguments");
  use_device(m);
  try {
    newton_solve(m, dt, &it, &cv);
  } catch (...) {
    if (niter) *niter = it;
    throw;
  }
  if (niter) *niter = it;
  if (converged) *converged = cv;
  SHAKTI_CATCH
}
int shakti_update_q(shakti_model* m) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(m, "null model");
  use_device(m);
  update_q(m);
  SHAKTI_CATCH
}
int shakti_update_melt(shakti_model* m) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(m, "null model");
  use_device(m);
  update_melt(m);
  SHAKTI_CATCH
}
int shakti_update_q_melt(shakti_model* m) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(m, "null model");
  use_device(m);
  update_q_melt(m);
  SHAKTI_CATCH
}
int shakti_update_b(shakti_model* m, double dt) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(m && dt > 0, "bad arguments");
  use_device(m);
  update_b(m, dt);
  SHAKTI_CATCH
}
int shakti_copy_N_to_N_n(shakti_model* m) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(m, "null model");
  use_device(m);
  copy_N(m);
  SHAKTI_CATCH
}
int shakti_step(shakti_model* m, double dt, int32_t* niter, int32_t* converged) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(m, "null model");
  use_device(m);
  shakti::step(m, dt, niter, converged);
  SHAKTI_CATCH
}
int shakti_run(shakti_model* m, const double* dts, int64_t nsteps, int32_t* niter_out) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(m && dts && nsteps >= 0, "bad arguments");
  use_device(m);
  require_diag_rows(m, nsteps);
  for (int64_t i = 0; i < nsteps; ++i) {
    int32_t it = 0, cv = 0;
    shakti::step(m, dts[i], &it, &cv);
    if (niter_out) niter_out[i] = it;
  }
  SHAKTI_CUDA(cudaStreamSynchronize(m->stream));
  SHAKTI_CATCH
}

int shakti_run_timed(shakti_model* m, const double* dts, int64_t nsteps, int32_t* niter_out, double* ms) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(m && dts && nsteps >= 0 && ms, "bad arguments");
  use_device(m);
  require_diag_rows(m, nsteps);
  cudaEvent_t e0, e1;
  SHAKTI_CUDA(cudaEventCreate(&e0));
  SHAKTI_CUDA(cudaEventCreate(&e1));
  SHAKTI_CUDA(cudaStreamSynchronize(m->stream));
  SHAKTI_CUDA(cudaEventRecord(e0, m->stream));
  for (int64_t i = 0; i < nsteps; ++i) {
    int32_t it = 0, cv = 0;
    shakti::step(m, dts[i], &it, &cv);
    if (niter_out) niter_out[i] = it;
  }
  SHAKTI_CUDA(cudaEventRecord(e1, m->stream));
  SHAKTI_CUDA(cudaEventSynchronize(e1));
  float t = 0;
  SHAKTI_CUDA(cudaEventElapsedTime(&t, e0, e1));
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  *ms = (double)t;
  SHAKTI_CATCH
}

int shakti_step_host(shakti_model* m, double dt, const double* inputs_host, double* b_out, double* N_out,
                     double* qx_out, double* qy_out, int32_t* niter, int32_t* converged) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(m, "null model");
  use_device(m);
  if (inputs_host) shakti::set_field(m, SHAKTI_F_INPUTS, inputs_host, 0);
  shakti::step(m, dt, niter, converged);
  if (b_out) shakti::get_field(m, SHAKTI_F_B, b_out, 0);
  if (N_out) shakti::get_field(m, SHAKTI_F_N, N_out, 0);
  if (qx_out) shakti::get_field(m, SHAKTI_F_QX, qx_out, 0);
  if (qy_out) shakti::get_field(m, SHAKTI_F_QY, qy_out, 0);
  SHAKTI_CATCH
}

int shakti_snapshot(shakti_model* m) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(m, "null model");
  use_device(m);
  const size_t nl = std::max<int32_t>(m->hm.n_local, 1);
  const double* src[6] = {m->N.p, m->N_n.p, m->b.p, m->qx.p, m->qy.p, m->melt.p};
  for (int k = 0; k < 6; ++k) {
    if (m->snap[k].n < nl) m->snap[k].alloc(nl);
    SHAKTI_CUDA(cudaMemcpyAsync(m->snap[k].p, src[k], sizeof(double) * nl, cudaMemcpyDeviceToDevice, m->stream));
  }
  m->snap_hist_ratio = m->hist_ratio; m->snap_hist_dt = m->hist_dt; m->snap_residual0 = m->residual0;
  m->snap_steps = m->st.steps;
  m->snap_t_model = m->t_model;
  m->snap_diag_n = m->diag_n;
  m->snap_valid = true;
  SHAKTI_CATCH
}

int shakti_rollback(shakti_model* m) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(m && m->snap_valid, "no snapshot to roll back to");
  use_device(m);
  const size_t nl = std::max<int32_t>(m->hm.n_local, 1);
  double* dst[6] = {m->N.p, m->N_n.p, m->b.p, m->qx.p, m->qy.p, m->melt.p};
  for (int k = 0; k < 6; ++k)
    SHAKTI_CUDA(cudaMemcpyAsync(dst[k], m->snap[k].p, sizeof(double) * nl, cudaMemcpyDeviceToDevice, m->stream));
  m->hist_ratio = m->snap_hist_ratio; m->hist_dt = m->snap_hist_dt; m->residual0 = m->snap_residual0;
  // the step counter goes back too, and the AMG hierarchy (numbers of a later state) is renewed at the next solve
  m->st.steps = m->snap_steps;
  m->t_model = m->snap_t_model;
  m->step_of_refresh = -1000000;
  m->diag_n = std::min(m->diag_n, m->snap_diag_n);   // records of the undone solves
  SHAKTI_CATCH
}

int shakti_diagnostics(shakti_model* m, double dt, double out[SHAKTI_D_COUNT]) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(m && out && dt > 0, "bad arguments");
  use_device(m);
  compute_kbar(m);
  assemble(m, dt, 0);
  const double r = norm2(m, m->F.p);
  double* row = m->diag_vals.p + kDiagVals;
  diagnostics_record(m, dt, 0, r, row);
  SHAKTI_CUDA(cudaMemcpyAsync(out, row, sizeof(double) * SHAKTI_D_COUNT, cudaMemcpyDeviceToHost, m->stream));
  SHAKTI_CUDA(cudaStreamSynchronize(m->stream));
  SHAKTI_CATCH
}

int shakti_record_diagnostics(shakti_model* m, int64_t capacity) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(m && capacity >= 0 && capacity <= ((int64_t)1 << 40), "bad arguments");
  use_device(m);
  SHAKTI_CUDA(cudaStreamSynchronize(m->stream));
  if (capacity > 0) m->diag_rows.alloc((size_t)capacity * SHAKTI_D_COUNT);
  else m->diag_rows.release();
  m->diag_cap = capacity;
  m->diag_n = m->snap_diag_n = 0;
  SHAKTI_CATCH
}

int shakti_read_diagnostics(shakti_model* m, double* rows, int64_t max_rows, int64_t* n_rows) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(m && n_rows, "null argument");
  *n_rows = m->diag_n;
  if (!rows) return SHAKTI_OK;
  SHAKTI_REQUIRE(max_rows >= m->diag_n, "row buffer too small for the recorded diagnostics");
  use_device(m);
  if (m->diag_n)
    SHAKTI_CUDA(cudaMemcpyAsync(rows, m->diag_rows.p, sizeof(double) * SHAKTI_D_COUNT * m->diag_n, cudaMemcpyDeviceToHost,
                                m->stream));
  SHAKTI_CUDA(cudaStreamSynchronize(m->stream));
  m->diag_n = m->snap_diag_n = 0;
  SHAKTI_CATCH
}

int shakti_set_moulins(shakti_model* m, int64_t n_moulins, const int32_t* vertex, const int64_t* knot_ptr,
                       const double* t_knots, const double* q_knots, double period) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(m, "null model");
  use_device(m);
  shakti::set_moulins(m, n_moulins, vertex, knot_ptr, t_knots, q_knots, period);
  SHAKTI_CATCH
}

int shakti_set_time(shakti_model* m, double t) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(m && std::isfinite(t), "bad arguments: the model time must be finite");
  m->t_model = t;
  SHAKTI_CATCH
}

int shakti_get_time(shakti_model* m, double* t) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(m && t, "null argument");
  *t = m->t_model;
  SHAKTI_CATCH
}

int shakti_moulin_discharge(shakti_model* m, double t, double* q_out) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(m && std::isfinite(t) && (q_out || m->n_moulins == 0), "bad arguments");
  for (int64_t k = 0; k < m->n_moulins; ++k) {
    const int64_t a = m->mo_kptr[k];
    q_out[k] = hydrograph_at(m->mo_t.data() + a, m->mo_q.data() + a, m->mo_kptr[k + 1] - a, m->mo_period, t);
  }
  SHAKTI_CATCH
}

// ---- model_setup data ingestion on the device (SURVEY row f3): the grid / polygon comes from the host, the
// mesh nodes are the model's own (already resident), the result lands directly in a vertex field
int shakti_interp_grid_to_field(shakti_model* m, int field, int32_t nx, int32_t ny, const double* xg, const double* yg,
                                const double* f_yx) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(m && xg && yg && f_yx && nx >= 2 && ny >= 2, "bad grid arguments");
  SHAKTI_REQUIRE(field >= 0 && field < SHAKTI_F_COUNT && field != SHAKTI_F_RESIDUAL, "field is not writable");
  use_device(m);
  DevBuf<double> dx, dy, df;
  dx.upload(xg, (size_t)nx);
  dy.upload(yg, (size_t)ny);
  df.upload(f_yx, (size_t)nx * ny);
  launch_interp_grid(m->hm.n_local, m->x.p, m->y.p, nx, ny, dx.p, dy.p, df.p, field_ptr(m, field), m->stream);
  if (field == SHAKTI_F_Z_B || field == SHAKTI_F_Z_S) m->h0_dirty = true;
  if (field != SHAKTI_F_INPUTS) m->hist_ratio = -1.0;
  SHAKTI_CUDA(cudaStreamSynchronize(m->stream));
  SHAKTI_CATCH
}

int shakti_polygon_to_field(shakti_model* m, int field, int32_t n_poly, const double* poly_xy) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(m && poly_xy && n_poly >= 3, "a polygon needs at least 3 vertices");
  SHAKTI_REQUIRE(field >= 0 && field < SHAKTI_F_COUNT && field != SHAKTI_F_RESIDUAL, "field is not writable");
  use_device(m);
  DevBuf<double> dp;
  dp.upload(poly_xy, (size_t)2 * n_poly);
  launch_points_in_polygon(m->hm.n_local, m->x.p, m->y.p, n_poly, dp.p, field_ptr(m, field), m->stream);
  if (field != SHAKTI_F_INPUTS) m->hist_ratio = -1.0;
  SHAKTI_CUDA(cudaStreamSynchronize(m->stream));
  SHAKTI_CATCH
}

// the same two operations for arbitrary points, without a model (host arrays in and out)
int shakti_interp_grid(int64_t n, const double* px, const double* py, int32_t nx, int32_t ny, const double* xg,
                       const double* yg, const double* f_yx, double* out) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(n >= 0 && px && py && xg && yg && f_yx && out && nx >= 2 && ny >= 2, "bad arguments");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    throw Error(SHAKTI_ERR_NO_DEVICE, "no CUDA device: the SHAKTI B200 path has no CPU fallback");
  }
  DevBuf<double> dpx, dpy, dx, dy, df, dout;
  dpx.upload(px, (size_t)n); dpy.upload(py, (size_t)n);
  dx.upload(xg, (size_t)nx); dy.upload(yg, (size_t)ny); df.upload(f_yx, (size_t)nx * ny);
  dout.alloc((size_t)std::max<int64_t>(n, 1));
  launch_interp_grid(n, dpx.p, dpy.p, nx, ny, dx.p, dy.p, df.p, dout.p, 0);
  SHAKTI_CUDA(cudaStreamSynchronize(0));
  if (n) SHAKTI_CUDA(cudaMemcpy(out, dout.p, sizeof(double) * n, cudaMemcpyDeviceToHost));
  SHAKTI_CATCH
}

int shakti_points_in_polygon(int64_t n, const double* px, const double* py, int32_t n_poly, const double* poly_xy,
                             double* out) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(n >= 0 && px && py && poly_xy && out && n_poly >= 3, "bad arguments");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    throw Error(SHAKTI_ERR_NO_DEVICE, "no CUDA device: the SHAKTI B200 path has no CPU fallback");
  }
  DevBuf<double> dpx, dpy, dp, dout;
  dpx.upload(px, (size_t)n); dpy.upload(py, (size_t)n);
  dp.upload(poly_xy, (size_t)2 * n_poly);
  dout.alloc((size_t)std::max<int64_t>(n, 1));
  launch_points_in_polygon(n, dpx.p, dpy.p, n_poly, dp.p, dout.p, 0);
  SHAKTI_CUDA(cudaStreamSynchronize(0));
  if (n) SHAKTI_CUDA(cudaMemcpy(out, dout.p, sizeof(double) * n, cudaMemcpyDeviceToHost));
  SHAKTI_CATCH
}

int shakti_wait_outputs(shakti_model* m) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(m, "null model");
  use_device(m);
  if (m->d2h_pending) {
    SHAKTI_CUDA(cudaEventSynchronize(m->ev_d2h));
    m->d2h_pending = false;
  }
  SHAKTI_CATCH
}

int shakti_step_host_async(shakti_model* m, double dt, const double* inputs_host, double* b_out, double* N_out,
                           double* qx_out, double* qy_out, int owned_only, int32_t* niter, int32_t* converged) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(m, "null model");
  use_device(m);
  const HostMesh& hm = m->hm;
  if (inputs_host) {
    if (owned_only) {
      // this rank's entries, in shakti_get_owned order, straight into the field; ghosts from their owners
      SHAKTI_CUDA(cudaMemcpyAsync(m->inputs.p, inputs_host, sizeof(double) * hm.n_owned, cudaMemcpyHostToDevice, m->stream));
      m->halo.exchange(m->inputs.p, m->stream);
    } else {
      SHAKTI_CUDA(cudaMemcpyAsync(m->stage.p, inputs_host, sizeof(double) * hm.nv_g, cudaMemcpyHostToDevice, m->stream));
      scatter_in(m, m->stage.p, m->inputs.p);
    }
  }
  shakti::step(m, dt, niter, converged);
  shakti::save_outputs_async(m, b_out, N_out, qx_out, qy_out, owned_only);
  SHAKTI_CATCH
}

int shakti_save_outputs_async(shakti_model* m, double* b_out, double* N_out, double* qx_out, double* qy_out,
                              int owned_only) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(m, "null model");
  use_device(m);
  shakti::save_outputs_async(m, b_out, N_out, qx_out, qy_out, owned_only);
  SHAKTI_CATCH
}

// Diagnostic: bandwidth of cudaMemcpyAsync between `host` (any host pointer) and a scratch device buffer,
// timed with CUDA events on a private stream, and the host time the enqueue itself takes (a pageable
// pointer makes the "async" call block while the driver stages the data).
int shakti_debug_copy_bw(void* host, int64_t bytes, int reps, double* h2d_gbs, double* d2h_gbs, double* enqueue_ms) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(host && bytes > 0 && reps > 0 && h2d_gbs && d2h_gbs && enqueue_ms, "bad arguments");
  void* dev = nullptr;
  SHAKTI_CUDA(cudaMalloc(&dev, (size_t)bytes));
  cudaStream_t st;
  SHAKTI_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
  cudaEvent_t e0, e1;
  SHAKTI_CUDA(cudaEventCreate(&e0));
  SHAKTI_CUDA(cudaEventCreate(&e1));
  for (int dir = 0; dir < 2; ++dir) {
    SHAKTI_CUDA(cudaStreamSynchronize(st));
    timespec t0, t1;
    SHAKTI_CUDA(cudaEventRecord(e0, st));
    clock_gettime(CLOCK_MONOTONIC, &t0);
    for (int i = 0; i < reps; ++i) {
      if (dir == 0) SHAKTI_CUDA(cudaMemcpyAsync(dev, host, (size_t)bytes, cudaMemcpyHostToDevice, st));
      else SHAKTI_CUDA(cudaMemcpyAsync(host, dev, (size_t)bytes, cudaMemcpyDeviceToHost, st));
    }
    clock_gettime(CLOCK_MONOTONIC, &t1);
    SHAKTI_CUDA(cudaEventRecord(e1, st));
    SHAKTI_CUDA(cudaEventSynchronize(e1));
    float ms = 0;
    SHAKTI_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    const double gbs = (double)bytes * reps / 1e9 / (ms / 1e3);
    if (dir == 0) { *h2d_gbs = gbs; enqueue_ms[0] = ((t1.tv_sec - t0.tv_sec) * 1e3 + (t1.tv_nsec - t0.tv_nsec) * 1e-6) / reps; }
    else { *d2h_gbs = gbs; enqueue_ms[1] = ((t1.tv_sec - t0.tv_sec) * 1e3 + (t1.tv_nsec - t0.tv_nsec) * 1e-6) / reps; }
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaStreamDestroy(st);
  cudaFree(dev);
  SHAKTI_CATCH
}

int shakti_alloc_pinned(int64_t bytes, void** out) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(out && bytes >= 0, "bad arguments");
  *out = nullptr;
  if (bytes) SHAKTI_CUDA(cudaMallocHost(out, (size_t)bytes));
  SHAKTI_CATCH
}
int shakti_free_pinned(void* p) {
  SHAKTI_TRY
  if (p) SHAKTI_CUDA(cudaFreeHost(p));
  SHAKTI_CATCH
}

int shakti_kernel_bytes(shakti_model* m, int which, double* bytes) {
  if (!m || !bytes) return SHAKTI_ERR_INVALID;
  const double nv = (double)m->hm.n_local, no = (double)m->hm.n_owned, ne = (double)m->hm.ne, nnz = (double)m->hm.A.nnz();
  switch (which) {
    case 0: *bytes = 12.0 * nnz + 20.0 * no; break;                                    // SpMV
    case 1: *bytes = 12.0 * ne + 8.0 * 12.0 * nv + 8.0 * ne + 8.0 * nnz + 8.0 * no; break;  // F+J assembly
    case 2: *bytes = 12.0 * ne + 8.0 * 5.0 * nv + 8.0 * ne; break;                      // Kbar
    case 3: *bytes = 12.0 * ne + 8.0 * 13.0 * nv; break;                                // nodal updates
    case 4: *bytes = 16.0 * no; break;                                                  // dot
    case 5: *bytes = 24.0 * no; break;                                                  // axpy
    default: return SHAKTI_ERR_INVALID;
  }
  return SHAKTI_OK;
}

int shakti_time_kernel(shakti_model* m, int which, int reps, double dt, double* ms_per_launch) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(m && ms_per_launch && reps > 0, "bad arguments");
  use_device(m);
  refresh_h0(m);
  cudaEvent_t e0, e1;
  SHAKTI_CUDA(cudaEventCreate(&e0));
  SHAKTI_CUDA(cudaEventCreate(&e1));
  auto once = [&]() {
    switch (which) {
      case 0: launch_spmv(view(m->J), m->dx.p, m->rhs.p, m->stream); break;
      case 1: assemble(m, dt, 1); break;
      case 2: compute_kbar(m); break;
      case 3:
        // the two kernels of a step's nodal pass (q + melt fused, then b), all outputs to scratch
        // vectors so the state is untouched
        launch_update_q_melt(m->hm.n_owned, m->win.p, m->x.p, m->y.p, m->h0.p, m->N.p, m->b.p, m->dx.p, m->rhs.p, m->G.p, m->melt.p, m->melt2.p, m->dprm, m->stream);
        launch_update_b(m->hm.n_owned, m->win.p, m->x.p, m->y.p, m->h0.p, m->N.p, m->b.p, m->qx.p, m->qy.p, m->G.p, m->melt.p, m->b2.p, dt, m->opt.b_min, m->dprm, m->stream);
        break;
      case 4: launch_multi_dot(m->red, m->hm.n_owned, 1, m->dx.p, m->hm.n_owned, m->rhs.p, m->scal.p, m->stream); break;
      case 5: launch_axpy(m->hm.n_owned, 0.0, m->dx.p, m->rhs.p, m->stream); break;
      default: throw Error(SHAKTI_ERR_INVALID, "unknown kernel id");
    }
  };
  if (which == 0) SHAKTI_REQUIRE(m->J_valid, "no assembled Jacobian");
  if (which == 1) compute_kbar(m);
  once();
  SHAKTI_CUDA(cudaEventRecord(e0, m->stream));
  for (int i = 0; i < reps; ++i) once();
  SHAKTI_CUDA(cudaEventRecord(e1, m->stream));
  SHAKTI_CUDA(cudaEventSynchronize(e1));
  float ms = 0;
  SHAKTI_CUDA(cudaEventElapsedTime(&ms, e0, e1));
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  *ms_per_launch = (double)ms / reps;
  SHAKTI_CATCH
}

int shakti_time_amg_smoother(shakti_model* m, int level, int reps, double* ms_per_launch, int64_t* rows, int64_t* nnz,
                             int32_t* value_bytes, int32_t* vector_bytes) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(m && ms_per_launch && reps > 0, "bad arguments");
  use_device(m);
  SHAKTI_REQUIRE(m->amg && m->amg->ready() && m->J_valid, "no AMG hierarchy yet: run a step first");
  int64_t r = 0, z = 0;
  int vb = 0;
  SHAKTI_REQUIRE(m->amg->launch_level_smoother(level, m->J, &r, &z, &vb), "no such AMG level on this rank");
  cudaEvent_t e0, e1;
  SHAKTI_CUDA(cudaEventCreate(&e0));
  SHAKTI_CUDA(cudaEventCreate(&e1));
  SHAKTI_CUDA(cudaEventRecord(e0, m->stream));
  for (int i = 0; i < reps; ++i) m->amg->launch_level_smoother(level, m->J, nullptr, nullptr);
  SHAKTI_CUDA(cudaEventRecord(e1, m->stream));
  SHAKTI_CUDA(cudaEventSynchronize(e1));
  float ms = 0;
  SHAKTI_CUDA(cudaEventElapsedTime(&ms, e0, e1));
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  *ms_per_launch = (double)ms / reps;
  if (rows) *rows = r;
  if (nnz) *nnz = z;
  if (value_bytes) *value_bytes = vb;
  if (vector_bytes) *vector_bytes = m->amg->fp32() ? 4 : 8;
  SHAKTI_CATCH
}

int shakti_time_amg_level_kernel(shakti_model* m, int level, int which, int reps, double* ms_per_launch, int64_t info[7]) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(m && ms_per_launch && info && reps > 0, "bad arguments");
  use_device(m);
  SHAKTI_REQUIRE(m->amg && m->amg->ready() && m->J_valid, "no AMG hierarchy yet: run a step first");
  SHAKTI_REQUIRE(m->amg->launch_level_kernel(level, which, m->J, info), "no such AMG level kernel on this rank");
  cudaEvent_t e0, e1;
  SHAKTI_CUDA(cudaEventCreate(&e0));
  SHAKTI_CUDA(cudaEventCreate(&e1));
  SHAKTI_CUDA(cudaEventRecord(e0, m->stream));
  for (int i = 0; i < reps; ++i) m->amg->launch_level_kernel(level, which, m->J, info);
  SHAKTI_CUDA(cudaEventRecord(e1, m->stream));
  SHAKTI_CUDA(cudaEventSynchronize(e1));
  float ms = 0;
  SHAKTI_CUDA(cudaEventElapsedTime(&ms, e0, e1));
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  *ms_per_launch = (double)ms / reps;
  SHAKTI_CATCH
}

// ---- AMG test hooks: one rank, where internal numbering = the rank's owned order
static void require_amg_hook(shakti_model* m, bool need_hierarchy) {
  SHAKTI_REQUIRE(m, "null model");
  SHAKTI_REQUIRE(!comm().active(), "the AMG test hooks run on one rank only");
  use_device(m);
  SHAKTI_REQUIRE(m->J_valid, "no assembled Jacobian");
  if (need_hierarchy) SHAKTI_REQUIRE(m->amg && m->amg->ready(), "no AMG hierarchy yet: call shakti_amg_refresh first");
}

int shakti_amg_refresh(shakti_model* m, int full) {
  SHAKTI_TRY
  require_amg_hook(m, false);
  ensure_amg(m);
  if (full) {
    m->amg->refresh(m->J, m->diag_pos.p);
    m->st.amg_refreshes++;
  } else {
    SHAKTI_REQUIRE(m->amg->ready(), "no AMG hierarchy to keep: refresh it in full first");
    m->amg->refresh_fine_smoother(m->J, m->diag_pos.p);
  }
  SHAKTI_CUDA(cudaStreamSynchronize(m->stream));
  SHAKTI_CATCH
}

int shakti_amg_level_info(shakti_model* m, int level, int64_t info[18]) {
  SHAKTI_TRY
  require_amg_hook(m, true);
  SHAKTI_REQUIRE(info, "null argument");
  SHAKTI_REQUIRE(m->amg->level_info(level, m->J, info), "no such AMG level");
  SHAKTI_CATCH
}

int shakti_amg_get_matrix(shakti_model* m, int level, int which, int32_t* rowptr, int32_t* col, double* val, int64_t* nnz) {
  SHAKTI_TRY
  require_amg_hook(m, true);
  SHAKTI_REQUIRE(nnz, "null argument");
  HostCsr a;
  std::vector<double> v;
  SHAKTI_REQUIRE(m->amg->level_matrix(level, which, m->J, a, v), "no such AMG level matrix");
  *nnz = a.nnz();
  if (rowptr) std::copy(a.rowptr.begin(), a.rowptr.end(), rowptr);
  if (col) std::copy(a.col.begin(), a.col.end(), col);
  if (val) std::copy(v.begin(), v.end(), val);
  SHAKTI_CATCH
}

int shakti_amg_get_vectors(shakti_model* m, int level, double* dinv, double* dinv_cycle, double* lmax, double* coef,
                           int32_t* stride) {
  SHAKTI_TRY
  require_amg_hook(m, true);
  std::vector<double> d, dc, c;
  double lm = 0.0;
  int st = 0;
  SHAKTI_REQUIRE(m->amg->level_vectors(level, d, dc, lm, c, st), "no such AMG level");
  if (dinv) std::copy(d.begin(), d.end(), dinv);
  if (dinv_cycle) std::copy(dc.begin(), dc.end(), dinv_cycle);
  if (lmax) *lmax = lm;
  if (coef) std::copy(c.begin(), c.end(), coef);
  if (stride) *stride = st;
  SHAKTI_CATCH
}

int shakti_amg_apply(shakti_model* m, const double* r, double* z) {
  SHAKTI_TRY
  require_amg_hook(m, true);
  SHAKTI_REQUIRE(r && z, "null argument");
  const int32_t no = m->hm.n_owned;
  SHAKTI_CUDA(cudaMemcpyAsync(m->rhs.p, r, sizeof(double) * no, cudaMemcpyHostToDevice, m->stream));
  SHAKTI_CUDA(cudaMemsetAsync(m->dx.p, 0, sizeof(double) * m->hm.n_local, m->stream));
  m->amg->apply(m->J, m->rhs.p, m->dx.p);
  SHAKTI_CUDA(cudaMemcpyAsync(z, m->dx.p, sizeof(double) * no, cudaMemcpyDeviceToHost, m->stream));
  SHAKTI_CUDA(cudaStreamSynchronize(m->stream));
  SHAKTI_CATCH
}

int shakti_comm_unique_id(uint8_t id[128]) {
  SHAKTI_TRY
  comm_unique_id(id);
  SHAKTI_CATCH
}
int shakti_comm_init(const uint8_t id[128], int rank, int nranks, int device) {
  SHAKTI_TRY
  comm_init(id, rank, nranks, device);
  SHAKTI_CATCH
}
int shakti_comm_finalize(void) {
  SHAKTI_TRY
  comm_finalize();
  SHAKTI_CATCH
}
int shakti_host_heap_selftest(int64_t heap_bytes, int32_t rounds, int32_t* violations) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(heap_bytes >= 4096 && rounds > 0 && violations, "bad arguments");
  *violations = heap_selftest((size_t)heap_bytes, rounds);
  SHAKTI_CATCH
}
int shakti_get_owned(shakti_model* m, int32_t* ids, int64_t* n_owned) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(m && n_owned, "null argument");
  *n_owned = m->hm.n_owned;
  if (ids) std::copy(m->hm.l2g.begin(), m->hm.l2g.begin() + m->hm.n_owned, ids);
  SHAKTI_CATCH
}

// ---------------------------------------------------------------- host-side helpers
struct shakti_host_mesh {
  shakti::HostMesh hm;
  shakti::AssemblyBlocks ab;
  bool ab_built = false;
};

// the host-only entry points take caller data that no shakti_create has looked at yet
static void require_valid_cells(int64_t n_vert, int64_t n_cell, const int32_t* cells) {
  SHAKTI_REQUIRE(n_vert > 0 && n_cell > 0 && n_vert <= 2000000000LL && n_cell <= 2000000000LL / 3, "mesh size out of range");
  for (int64_t i = 0; i < 3 * n_cell; ++i)
    SHAKTI_REQUIRE(cells[i] >= 0 && cells[i] < n_vert, "cell vertex id out of range");
}

int shakti_host_csr_pattern(int64_t n_vert, int64_t n_cell, const int32_t* cells, int32_t* rowptr, int32_t* col,
                            int64_t* nnz) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(cells && nnz && n_vert > 0 && n_cell > 0, "bad arguments");
  require_valid_cells(n_vert, n_cell, cells);
  HostCsr a = caller_csr(n_vert, n_cell, cells);
  *nnz = a.nnz();
  if (rowptr) std::copy(a.rowptr.begin(), a.rowptr.end(), rowptr);
  if (col) std::copy(a.col.begin(), a.col.end(), col);
  SHAKTI_CATCH
}
int shakti_host_locate_dirichlet(int64_t n_vert, int64_t n_cell, const int32_t* cells, const uint8_t* marker,
                                 int32_t* dofs, int64_t cap, int64_t* n_out) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(cells && marker && n_out, "null argument");
  require_valid_cells(n_vert, n_cell, cells);
  std::vector<int32_t> d = locate_dirichlet_dofs(n_vert, n_cell, cells, marker);
  *n_out = (int64_t)d.size();
  if (dofs) {
    SHAKTI_REQUIRE(cap >= (int64_t)d.size(), "dof buffer too small");
    std::copy(d.begin(), d.end(), dofs);
  }
  SHAKTI_CATCH
}
int shakti_host_mesh_create(int64_t n_vert, int64_t n_cell, const double* xy, const int32_t* cells, int rank,
                            int nranks, int reorder, shakti_host_mesh** out) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(xy && cells && out && nranks >= 1 && rank >= 0 && rank < nranks, "bad arguments");
  std::unique_ptr<shakti_host_mesh> h(new shakti_host_mesh());
  build_host_mesh(n_vert, n_cell, xy, cells, rank, nranks, reorder, h->hm);
  *out = h.release();
  SHAKTI_CATCH
}
int shakti_host_mesh_destroy(shakti_host_mesh* hm) {
  delete hm;
  return SHAKTI_OK;
}
int shakti_host_mesh_info(shakti_host_mesh* h, int64_t info[6]) {
  if (!h || !info) return SHAKTI_ERR_INVALID;
  info[0] = h->hm.n_owned; info[1] = h->hm.n_local; info[2] = h->hm.ne; info[3] = h->hm.A.nnz();
  info[4] = h->hm.S.padded(); info[5] = (int64_t)h->hm.nbrs.size();
  return SHAKTI_OK;
}
int shakti_host_mesh_array(shakti_host_mesh* h, int which, int32_t* out, int64_t* n) {
  SHAKTI_TRY
  SHAKTI_REQUIRE(h && n, "null argument");
  const HostMesh& m = h->hm;
  std::vector<int32_t> tmp;
  const std::vector<int32_t>* v = nullptr;
  switch (which) {
    case SHAKTI_HM_L2G: v = &m.l2g; break;
    case SHAKTI_HM_CELLS: v = &m.cells; break;
    case SHAKTI_HM_CELL_L2G: v = &m.cell_l2g; break;
    case SHAKTI_HM_ROWPTR: v = &m.A.rowptr; break;
    case SHAKTI_HM_COL: v = &m.A.col; break;
    case SHAKTI_HM_SLICE_PTR: v = &m.S.slice_ptr; break;
    case SHAKTI_HM_SELL_COL: v = &m.S.col; break;
    case SHAKTI_HM_SLOT: v = &m.slot; break;
    case SHAKTI_HM_DIAG_POS: v = &m.diag_pos; break;
    case SHAKTI_HM_WIN: v = &m.win; break;
    case SHAKTI_HM_WIN_CELL: v = &m.win_cell; break;
    case SHAKTI_HM_CELL_COUNTED: v = &m.cell_counted; break;
    case SHAKTI_HM_NBR_RANK:
      for (const auto& nb : m.nbrs) tmp.push_back(nb.rank);
      v = &tmp; break;
    case SHAKTI_HM_NBR_SEND_PTR:
      tmp.push_back(0);
      for (const auto& nb : m.nbrs) tmp.push_back(tmp.back() + (int32_t)nb.send_local.size());
      v = &tmp; break;
    case SHAKTI_HM_NBR_SEND_IDX:
      for (const auto& nb : m.nbrs) tmp.insert(tmp.end(), nb.send_local.begin(), nb.send_local.end());
      v = &tmp; break;
    case SHAKTI_HM_NBR_RECV:
      for (const auto& nb : m.nbrs) { tmp.push_back(nb.recv_begin); tmp.push_back(nb.recv_count); }
      v = &tmp; break;
    case SHAKTI_HM_AB_INFO: case SHAKTI_HM_AB_EPTR: case SHAKTI_HM_AB_ELEMS: case SHAKTI_HM_AB_LV: case SHAKTI_HM_AB_HPTR:
    case SHAKTI_HM_AB_HALO: case SHAKTI_HM_AB_INCPTR: case SHAKTI_HM_AB_INC: case SHAKTI_HM_AB_SRC: {
      if (!h->ab_built) { build_assembly_blocks(m, 400, h->ab); h->ab_built = true; }
      const AssemblyBlocks& ab = h->ab;
      switch (which) {
        case SHAKTI_HM_AB_INFO: tmp = {ab.rows_per_block, ab.n_blocks, ab.max_cells, ab.max_verts, ab.ok ? 1 : 0}; break;
        case SHAKTI_HM_AB_EPTR: tmp = ab.blk_eptr; break;
        case SHAKTI_HM_AB_ELEMS: tmp = ab.blk_elems; break;
        case SHAKTI_HM_AB_LV: tmp.assign(ab.blk_lv.begin(), ab.blk_lv.end()); break;
        case SHAKTI_HM_AB_HPTR: tmp = ab.blk_hptr; break;
        case SHAKTI_HM_AB_HALO: tmp = ab.blk_halo; break;
        case SHAKTI_HM_AB_INCPTR: tmp = ab.inc_ptr; break;
        case SHAKTI_HM_AB_INC: tmp.assign(ab.inc_code.begin(), ab.inc_code.end()); break;
        default: tmp.resize(ab.src.size()); std::memcpy(tmp.data(), ab.src.data(), ab.src.size() * sizeof(uint32_t)); break;
      }
      v = &tmp; break;
    }
    default: throw Error(SHAKTI_ERR_INVALID, "unknown host array id");
  }
  if (out) {
    SHAKTI_REQUIRE(*n >= (int64_t)v->size(), "array buffer too small");
    std::copy(v->begin(), v->end(), out);
  }
  *n = (int64_t)v->size();
  SHAKTI_CATCH
}

}  // extern "C"
