/* shakti_b200.h — C ABI of the B200-native SHAKTI transient solver.
 *
 * This is the drop-in boundary for the hot path of agstub/shakti-fenics: everything that
 * `source/solvers.py` delegates to DOLFINx / FFCx / Basix / PETSc per time step.  The
 * reference has no FFI of its own (it is pure Python over third-party native code), so each
 * entry point below names the reference call site(s) whose work it takes over; INTEGRATION.md
 * shows the ctypes binding a maintainer adds to `source/solvers.py`.
 *
 * Conventions
 *   - plain C: pointers + sizes, no torch/CUDA types.  Pointers are HOST pointers unless the
 *     `is_device` argument of a call says otherwise (then they are device pointers on the
 *     GPU the handle was created on, e.g. `tensor.data_ptr()`).
 *   - vertex (dof) and cell numbering in every argument is the CALLER's numbering (the
 *     reference assumes geometry node index == P1 dof index, model_setup.py:70-71); the
 *     library reorders internally and undoes it at this boundary.
 *   - every function returns 0 on success and a negative shakti_status on error;
 *     shakti_last_error() returns a human-readable message for the calling thread.
 *   - fp64 data, int32 indices.  There is no CPU fallback: without a usable sm_100 device
 *     shakti_create fails with SHAKTI_ERR_NO_DEVICE.
 */
#ifndef SHAKTI_B200_H
#define SHAKTI_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct shakti_model shakti_model;   /* opaque handle; owns all device memory */

typedef enum shakti_status {
  SHAKTI_OK = 0,
  SHAKTI_ERR_INVALID = -1,       /* bad argument */
  SHAKTI_ERR_NO_DEVICE = -2,     /* no CUDA device / wrong architecture */
  SHAKTI_ERR_CUDA = -3,          /* CUDA runtime error (message has the detail) */
  SHAKTI_ERR_NOT_CONVERGED = -4, /* Newton did not converge (reference: RuntimeError, solvers.py:179-180) */
  SHAKTI_ERR_LINEAR = -5,        /* Krylov solve failed to reach its tolerance */
  SHAKTI_ERR_COMM = -6           /* NCCL / multi-GPU set-up error */
} shakti_status;

/* source/params.py:4-11.  n is Glen's exponent (a Python int 3 there). */
typedef struct shakti_params {
  double g, rho_i, rho_w, nu, Lh, omega, n, A;
} shakti_params;

/* Vertex fields.  Inputs follow model_setup.py:44-51; state follows solvers.py:129-156. */
typedef enum shakti_field {
  SHAKTI_F_Z_B = 0,      /* md.z_b        bed elevation [m]                       */
  SHAKTI_F_Z_S = 1,      /* md.z_s        surface elevation [m]                   */
  SHAKTI_F_G = 2,        /* md.G          geothermal flux [W/m^2]                 */
  SHAKTI_F_INPUTS = 3,   /* md.inputs     water input [m/s]                       */
  SHAKTI_F_STORAGE = 4,  /* `storage` of solvers.py:147-152 (zeros or md.lake_bdry) */
  SHAKTI_F_B = 5,        /* b             gap height [m]                          */
  SHAKTI_F_N = 6,        /* N             effective pressure [Pa]                 */
  SHAKTI_F_N_N = 7,      /* N_n           N at previous step                      */
  SHAKTI_F_QX = 8,       /* q.sub(0)      water flux x [m^2/s]                    */
  SHAKTI_F_QY = 9,       /* q.sub(1)      water flux y                            */
  SHAKTI_F_MELT_N = 10,  /* melt_n        melt rate at previous step              */
  SHAKTI_F_RESIDUAL = 11,/* F of the last assembly (read-only)                    */
  SHAKTI_F_COUNT = 12
} shakti_field;

typedef enum shakti_linear_solver { SHAKTI_KSP_GMRES = 0, SHAKTI_KSP_BICGSTAB = 1 } shakti_linear_solver;
typedef enum shakti_precond { SHAKTI_PC_JACOBI = 0, SHAKTI_PC_AMG = 1, SHAKTI_PC_NONE = 2 } shakti_precond;
/* Denominator of NewtonSolver's relative test ||F||/r0 < rtol (solvers.py:52,179 [EXT]).
 * INITIAL_RESIDUAL (default): r0 = ||F||_2 at iteration 0 of the current solve (SURVEY.md row
 * a11).  DOLFINX: r0 = ||dx||_2 of iteration 1, never reset between solves and 0 before the very
 * first one -- what the DOLFINx 0.8/0.9 C++ class is believed to do; unverifiable offline, and
 * scale dependent (a time step is skipped whenever ||F|| < rtol * ||dx_1|| of the previous step). */
typedef enum shakti_newton_r0 {
  SHAKTI_R0_DOLFINX = 0,
  SHAKTI_R0_INITIAL_RESIDUAL = 1
} shakti_newton_r0;

/* Solver options.  Newton defaults are DOLFINx NewtonSolver's (solvers.py:52): rtol 1e-9,
 * atol 1e-10, max_it 50, relaxation 1.  The reference's linear solve is a direct LU; the
 * Krylov tolerance is therefore far below the Newton tolerance by default. */
typedef struct shakti_options {
  double newton_rtol, newton_atol;
  int32_t newton_max_it;
  int32_t newton_r0;            /* shakti_newton_r0 */
  int32_t linear_solver;        /* shakti_linear_solver */
  int32_t precond;              /* shakti_precond */
  double linear_rtol;           /* floor of the Krylov target: ||J dx - F_k|| <= linear_rtol * ||F_0|| (F_0: residual the Newton
                                   solve started from); see linear_forcing */
  double linear_atol;
  int32_t linear_max_it;
  int32_t gmres_restart;
  int32_t amg_refresh_every;    /* recompute AMG numerics at the first Newton solve of every k-th time step (>=1) */
  int32_t amg_max_levels;
  int32_t amg_coarse_size;      /* stop coarsening below this many rows */
  int32_t amg_presmooth, amg_postsmooth; /* Jacobi sweeps, or Chebyshev polynomial degree */
  double amg_smoother_omega;    /* damped-Jacobi weight on every level */
  double amg_prolong_omega;     /* prolongator smoothing weight (0 = plain aggregation) */
  double amg_strength_theta;    /* strong connection: |a_ij| >= theta 0.5^level sqrt(|a_ii a_jj|) (0 = all) */
  double amg_cheby_ratio;       /* Chebyshev smoothing interval [lmax/ratio, lmax] of D^-1 A */
  int32_t amg_smoother;         /* 0 = damped Jacobi, 1 = Chebyshev */
  int32_t amg_fp32_cycle;       /* 1 = V-cycle in single precision under FGMRES (set-up, Krylov, residuals stay fp64) */
  int32_t amg_cuda_graph;       /* 1 = on a single GPU the V-cycle is replayed as a captured CUDA graph */
  int32_t amg_smoother_halo;    /* multi-GPU: 1 = exchange ghosts before every smoothing step, 0 = only before the residual and the
                                   prolongation (ghosts lag inside the smoother: fewer messages, a slightly weaker preconditioner) */
  double b_min;                 /* md.b_min, model_setup.py:53 */
  int32_t assembly_kernel;      /* 0 = row-block staged gather (default), 1 = element atomics */
  int32_t reorder;              /* 1 = internal Morton reordering (default), 0 = keep caller order */
  double linear_forcing;        /* > 0 (default 0.01): the Krylov solve of a Newton iteration stops at linear_forcing x the
                                   residual the NEXT Newton iterate is predicted to have (never below linear_rtol ||F_0||, never
                                   above 1e-2 ||F_k||); 0 = always solve to linear_rtol ||F_0|| (closest to the reference's LU) */
  int32_t amg_replicate_below;  /* multi-GPU: the first AMG level with at most this many rows in total, and every level below
                                   it, is replicated on all ranks and solved without communication (default 100000) */
  double newton_relaxation;     /* DOLFINx NewtonSolver.relaxation_parameter: x <- x - relaxation * dx.  Default 1, which is what
                                   the reference runs with (solvers.py:52 leaves the attribute alone) */
  int32_t newton_line_search;   /* 0 (default) = the reference's plain Newton step.  k > 0 = backtracking line search on
                                   ||F||_2: the step length starts at newton_relaxation and is halved, at most k times, until
                                   ||F(x - s dx)|| <= (1 - 1e-4 s) ||F(x)|| (an extension named by BASELINE.json's north_star;
                                   DOLFINx has none).  A step that is accepted at full length costs nothing extra. */
} shakti_options;

typedef struct shakti_stats {
  int64_t n_vert, n_cell, nnz;          /* global sizes                                       */
  int64_t n_owned, n_local, n_cell_local, nnz_local;
  int64_t steps, newton_its, linear_its; /* cumulative since create / reset                   */
  int64_t kernel_launches;               /* kernels of this library launched since create      */
  int64_t amg_levels, amg_refreshes;
  double amg_operator_complexity;
  double last_residual, last_residual0;  /* Newton: ||F|| at exit and the r0 used               */
  double last_linear_relres;
  int64_t newton_backtracks;             /* step halvings taken by the line search (newton_line_search > 0) */
} shakti_stats;

/* ---------------------------------------------------------------- lifetime */

/* Fill `opt` with defaults. */
int shakti_default_options(shakti_options* opt);
int shakti_default_params(shakti_params* p);

/* Build a model on the current CUDA device (or `device` >= 0).
 * Replaces: functionspace/dofmap/sparsity-pattern creation and form compilation that DOLFINx
 * performs for model_setup.py:29-30 and solvers.py:51 (NonlinearProblem).
 *   xy    : n_vert x 2 (row-major) vertex coordinates  (domain.geometry.x[:,0:2])
 *   cells : n_cell x 3 (row-major) vertex ids per triangle (V.dofmap.list == geometry dofmap)
 * For multi-GPU runs call shakti_comm_init first on every rank and pass the same GLOBAL mesh
 * on every rank; the library keeps the rank's partition.
 * Every vertex must belong to at least one cell (DOLFINx drops unreferenced nodes when it builds a mesh):
 * a mesh with such a vertex is refused with SHAKTI_ERR_INVALID on every rank. */
int shakti_create(int64_t n_vert, int64_t n_cell, const double* xy, const int32_t* cells,
                  const shakti_params* params, const shakti_options* opt, int device,
                  shakti_model** out);
int shakti_destroy(shakti_model* m);
const char* shakti_last_error(void);
const char* shakti_version(void);
/* Number of CUDA devices visible to this process (0 without a driver / device). */
int shakti_device_count(int* n);

/* ---------------------------------------------------------------- data in / out */

/* Copy a whole vertex field in (caller numbering, n_vert doubles).  Replaces the
 * `Function.x.array[:] = ...` / `.interpolate(...)` writes of setups and solvers.py:137-140. */
int shakti_set_field(shakti_model* m, int field, const double* src, int is_device);
int shakti_get_field(shakti_model* m, int field, double* dst, int is_device);
/* Interleaved flux q = [qx0,qy0,qx1,...] (blocked vector-P1 layout of md.q_init / q). */
int shakti_set_flux(shakti_model* m, const double* q_interleaved, int is_device);
int shakti_get_flux(shakti_model* m, double* q_interleaved, int is_device);

/* model_setup data ingestion on the device (reference model_setup.py:68-91; SURVEY row f3).
 * shakti_interp_grid_to_field: bilinear interpolation (linear extrapolation outside the grid) of a gridded
 *   field f_yx[iy*nx + ix] given on ascending axes xg[nx], yg[ny] onto the mesh nodes, written straight into
 *   vertex field `field` -- RegularGridInterpolator((x, y), f.T, bounds_error=False, fill_value=None) of
 *   model_setup.interp_data, without the host round trip of the nodal array.
 * shakti_polygon_to_field: 1.0 at nodes inside the closed polygon poly_xy[n_poly][2] (even-odd rule), else 0.0
 *   -- the lake indicator of model_setup.set_lake_bdry.
 * The two functions without a model do the same for arbitrary host points (parity hooks). */
int shakti_interp_grid_to_field(shakti_model* m, int field, int32_t nx, int32_t ny, const double* xg, const double* yg,
                                const double* f_yx);
int shakti_polygon_to_field(shakti_model* m, int field, int32_t n_poly, const double* poly_xy);
int shakti_interp_grid(int64_t n, const double* px, const double* py, int32_t nx, int32_t ny, const double* xg,
                       const double* yg, const double* f_yx, double* out);
int shakti_points_in_polygon(int64_t n, const double* px, const double* py, int32_t n_poly, const double* poly_xy,
                             double* out);

/* Dirichlet dofs and value: solvers.py:17-26 (get_bcs).  n_dofs == 0 <=> outflow_on False. */
int shakti_set_dirichlet(shakti_model* m, const int32_t* dofs, int64_t n_dofs, double value);
/* Boundary facets whose vertices all satisfy marker[v] != 0 -> dofs; replaces
 * locate_entities_boundary + locate_dofs_topological (solvers.py:22-23).  Returns the count
 * and (if dofs != NULL, capacity cap) the sorted dof list. */
int shakti_locate_dirichlet(shakti_model* m, const uint8_t* marker, int32_t* dofs, int64_t cap,
                            int64_t* n_out);

/* Quadrature table used for the transmissivity integral (reference triangle, weights sum to
 * 1/2): the rule FFCx/Basix would pick for the forms of solvers.py:45,51.  Max 64 points. */
int shakti_set_quadrature(shakti_model* m, int32_t n_pts, const double* pts_xy, const double* wts);

int shakti_set_options(shakti_model* m, const shakti_options* opt);
int shakti_get_options(shakti_model* m, shakti_options* opt);
int shakti_get_stats(shakti_model* m, shakti_stats* st);

/* ---------------------------------------------------------------- parity hooks */

/* CSR pattern of the Jacobian in caller numbering (sorted unique columns, diagonal included):
 * what PETSc's MatAIJ holds for solvers.py:51.  Call with NULL arrays to query nnz. */
int shakti_get_csr(shakti_model* m, int32_t* rowptr, int32_t* col, int64_t* nnz);
/* Per-cell transmissivity integral Kbar_T (caller cell order), from the current b, q. */
int shakti_kbar(shakti_model* m, double* kbar_out);
/* One residual + Jacobian assembly at the current state (what NonlinearProblem.F/.J do for
 * solvers.py:179): F_out n_vert doubles, Jvals_out nnz doubles in shakti_get_csr order;
 * either may be NULL.  Dirichlet handling included. */
int shakti_assemble(shakti_model* m, double dt, double* F_out, double* Jvals_out);
/* y = J x with the last assembled Jacobian (host arrays, caller numbering). */
int shakti_spmv(shakti_model* m, const double* x, double* y);
/* Solve J dx = rhs with the configured Krylov method on the last assembled Jacobian. */
int shakti_linear_solve(shakti_model* m, const double* rhs, double* dx, int32_t* iters,
                        double* relres);
/* Winning cell (caller cell index) per vertex for Function.interpolate(Expression). */
int shakti_get_winning_cells(shakti_model* m, int32_t* win_cell);

/* ---------------------------------------------------------------- the hot path */

/* solvers.py:48  N.interpolate(N_n) — once, when the solver is built. */
int shakti_start(shakti_model* m);
/* solvers.py:179  niter, converged = solver.solve(N) */
int shakti_newton_solve(shakti_model* m, double dt, int32_t* niter, int32_t* converged);
/* solvers.py:186 / :189 / :192-197 */
int shakti_update_q(shakti_model* m);
int shakti_update_melt(shakti_model* m);
int shakti_update_b(shakti_model* m, double dt);
/* solvers.py:186 and :189 in one pass over the vertices (same results as the two calls above) */
int shakti_update_q_melt(shakti_model* m);
/* solvers.py:228-229 */
int shakti_copy_N_to_N_n(shakti_model* m);
/* Device-side snapshot of the time-dependent state (N, N_n, b, q, melt_n and the solver's convergence history)
 * and return to it: lets a caller retry a failed step with a smaller dt, or repeat the same steps (bench.py
 * measures the device-resident and the end-to-end rate over the SAME steps this way).  Extension: the
 * reference has nothing like it (solvers.py:168-229 only moves forward). */
int shakti_snapshot(shakti_model* m);
int shakti_rollback(shakti_model* m);
/* One whole pass of solvers.py:179-229 (without file output). */
int shakti_step(shakti_model* m, double dt, int32_t* niter, int32_t* converged);
/* nsteps passes with the given dt list; niter_out (nsteps int32) may be NULL. */
int shakti_run(shakti_model* m, const double* dts, int64_t nsteps, int32_t* niter_out);
/* shakti_run bracketed by CUDA events on the library's stream; *ms = device time of the nsteps
 * steps (the caller barriers/synchronises around it and takes the max over ranks). */
int shakti_run_timed(shakti_model* m, const double* dts, int64_t nsteps, int32_t* niter_out, double* ms);
/* Same as shakti_step with host buffers in the call: copies `inputs_host` (n_vert doubles,
 * may be NULL) to the device before the step and b, N, qx, qy (each n_vert doubles, any may
 * be NULL) back after it — the per-save traffic of solvers.py:199-208. */
int shakti_step_host(shakti_model* m, double dt, const double* inputs_host, double* b_out,
                     double* N_out, double* qx_out, double* qy_out, int32_t* niter,
                     int32_t* converged);

/* Asynchronous, double-buffered form of shakti_step_host (the save path of solvers.py:199-225 without
 * stalling the time loop).  The step itself is complete on return (niter / converged are final); the
 * device->host copies of b, N, qx, qy into the given buffers (pinned memory for true overlap; any may
 * be NULL) are only ENQUEUED on a second stream from on-device snapshots, so they overlap the next
 * step.  The buffers are valid after shakti_wait_outputs(); alternate two buffer sets to keep a step's
 * output while the next one runs.
 *   owned_only = 0: buffers hold n_vert doubles in caller numbering (other ranks' entries are 0);
 *   owned_only = 1: buffers (and inputs_host) hold this rank's n_owned doubles in shakti_get_owned order,
 *                   so N ranks move 1/N of the bytes each and the caller places them with that index map. */
int shakti_step_host_async(shakti_model* m, double dt, const double* inputs_host, double* b_out,
                           double* N_out, double* qx_out, double* qy_out, int owned_only,
                           int32_t* niter, int32_t* converged);
int shakti_wait_outputs(shakti_model* m);
/* The output half alone (for callers that drive the split entry points, as solvers.solve(md) does). */
int shakti_save_outputs_async(shakti_model* m, double* b_out, double* N_out, double* qx_out, double* qy_out,
                              int owned_only);
/* Page-locked host memory for those buffers (cudaMallocHost / cudaFreeHost). */
int shakti_alloc_pinned(int64_t bytes, void** out);
int shakti_free_pinned(void* p);
/* ---------------------------------------------------------------- water-budget diagnostics
 * One record of SHAKTI_D_COUNT doubles describes the state a Newton solve converged on: the new N with the
 * lagged b, q, melt_n and N_n the residual was built from (NOT the state after the nodal updates).  Integrals
 * use the assembly's own quadrature; every value is global (summed / reduced over ranks).  With F~ the residual
 * without Dirichlet replacement or lifting, sum_i F~_i = int R, which splits into the identity
 *   outflow = input - (1/rho_i - 1/rho_w) melt + closure + storage + imbalance
 * that holds at every converged step up to rounding (DESIGN.md, "Water-budget diagnostics").  With moulins,
 * sum_i F~_i = int R - sum_k Q_k(t), so the moulin discharge at the solve's time t = model time + dt is part of
 * `input` (each rank adds its own moulins). */
typedef enum shakti_diag {
  SHAKTI_D_DT = 0,          /* dt of the solve [s]                                          */
  SHAKTI_D_NEWTON_ITS = 1,  /* Newton iterations                                            */
  SHAKTI_D_RESIDUAL = 2,    /* ||F||_2 at exit (stats.last_residual)                        */
  SHAKTI_D_AREA = 3,        /* int 1 [m^2]                                                  */
  SHAKTI_D_WATER_VOLUME = 4,/* int b [m^3]                                                  */
  SHAKTI_D_INPUT = 5,       /* int inputs + sum_k Q_k(t) of the moulins [m^3/s] (no moulins: int inputs) */
  SHAKTI_D_MELT = 6,        /* int (m0 + mdiff) [kg/s]                                      */
  SHAKTI_D_CLOSURE = 7,     /* int A b N|N|^(n-1) [m^3/s]                                   */
  SHAKTI_D_STORAGE = 8,     /* int storage (N - N_n) / (rho_w g dt) [m^3/s]                 */
  SHAKTI_D_OUTFLOW = 9,     /* -sum over Dirichlet rows of F~: discharge through the boundary [m^3/s] */
  SHAKTI_D_IMBALANCE = 10,  /* sum over the other rows of F~ (moulin rows included): what Newton left [m^3/s] */
  SHAKTI_D_N_MEAN = 11,     /* int N / int 1 [Pa]                                           */
  SHAKTI_D_N_MIN = 12,      /* min over vertices [Pa]                                       */
  SHAKTI_D_N_MAX = 13,      /* max over vertices [Pa]                                       */
  SHAKTI_D_B_MAX = 14,      /* max over vertices [m]                                        */
  SHAKTI_D_COUNT = 15
} shakti_diag;
/* One record of the current state, synchronous (a parity hook): recomputes Kbar; columns 0-2 are dt, 0 and
 * ||F||_2 of the current state (the residual field is re-assembled). */
int shakti_diagnostics(shakti_model* m, double dt, double out[SHAKTI_D_COUNT]);
/* capacity > 0: every converged Newton solve (shakti_newton_solve, shakti_step, shakti_run*, shakti_step_host*)
 * appends one record to a device buffer of `capacity` rows, on the stream, without a host synchronisation.
 * 0 (the default): off, a step launches nothing extra.  Rows not yet read are discarded.  A solve that finds
 * the buffer full fails with SHAKTI_ERR_INVALID before it changes any state; shakti_run checks nsteps
 * against the free rows up front.  Rows recorded after shakti_snapshot are dropped by shakti_rollback. */
int shakti_record_diagnostics(shakti_model* m, int64_t capacity);
/* Copy the recorded rows (row-major, SHAKTI_D_COUNT doubles each; max_rows must hold them all) to `rows` and
 * empty the buffer; *n_rows = rows copied.  rows == NULL: only query the count (the buffer is kept). */
int shakti_read_diagnostics(shakti_model* m, double* rows, int64_t max_rows, int64_t* n_rows);

/* ---------------------------------------------------------------- moulins (point water inputs)
 * Extension: the reference's only water input is the distributed field md.inputs (solvers.py:45).  A moulin is a
 * caller vertex v_k with a piecewise-linear hydrograph Q_k(t) [m^3/s]: knots (t_j, Q_j) with t_j strictly
 * increasing, linear between knots, constant outside them.  period > 0 first wraps t into [t_0, t_0 + period) of
 * each hydrograph (diurnal cycles); 0 means no period.  After every assembly
 *   F_i -= sum over k with v_k = i of Q_k(t)       (moulins of one vertex summed in the order given, no atomics)
 * -- the source term of solvers.py:45 with a Dirac right-hand side, the sign of the `- inputs` term.  The Jacobian
 * is unchanged.  The model keeps a clock: a Newton solve (and shakti_assemble / shakti_diagnostics) with step dt
 * evaluates Q at model time + dt, the end of the step; shakti_update_b (which closes a step) advances the clock
 * by dt; shakti_snapshot / shakti_rollback save and restore it.  It starts at 0.
 * A moulin may not sit on a Dirichlet dof: shakti_set_moulins refuses one, and so does a later
 * shakti_set_dirichlet that would create one.  On several GPUs every rank passes the same (global) list; each rank
 * applies the moulins of the vertices it owns.  Without moulins a step launches exactly what it did before. */
/* n_moulins moulins: vertex[k] (caller id); the knots of moulin k are t_knots / q_knots [knot_ptr[k],
 * knot_ptr[k+1]), knot_ptr[0] = 0 (n_moulins + 1 entries).  Replaces the previous set; n_moulins = 0 removes all.
 * Invalid arguments (vertex out of range or on a Dirichlet dof, an empty hydrograph, non-increasing knot times,
 * NaN or Inf, a negative period) return SHAKTI_ERR_INVALID and leave the model unchanged. */
int shakti_set_moulins(shakti_model* m, int64_t n_moulins, const int32_t* vertex, const int64_t* knot_ptr,
                       const double* t_knots, const double* q_knots, double period);
/* The model clock [s] (finite). */
int shakti_set_time(shakti_model* m, double t);
int shakti_get_time(shakti_model* m, double* t);
/* Parity hook: q_out[k] = Q_k(t) in caller order, evaluated on the host with the device's arithmetic. */
int shakti_moulin_discharge(shakti_model* m, double t, double* q_out);

/* Diagnostic: GB/s of cudaMemcpyAsync host->device / device->host for `host` (any host pointer) and the host
 * milliseconds each enqueue took (enqueue_ms[0] h2d, [1] d2h): tells page-locked from pageable memory. */
int shakti_debug_copy_bw(void* host, int64_t bytes, int reps, double* h2d_gbs, double* d2h_gbs, double* enqueue_ms);

/* ---------------------------------------------------------------- micro-benchmarks
 * Launch one kernel `reps` times on the library stream and return the mean device time per
 * launch in milliseconds (CUDA events on that stream).  `which`: 0 = SpMV (fine Jacobian),
 * 1 = F+J assembly, 2 = Kbar, 3 = nodal updates (q, melt, b), 4 = dot, 5 = axpy. */
int shakti_time_kernel(shakti_model* m, int which, int reps, double dt, double* ms_per_launch);
/* One smoothing step of AMG level `level` (the V-cycle's dominant kernel: SELL SpMV fused with the Chebyshev
 * recurrence, in the cycle's precision), timed the same way.  Returns the level's local rows and stored
 * entries, the bytes per matrix value (2: half-precision row-scaled copy on the large levels, 4: fp32 copy) and
 * per vector entry, from which the caller forms the algorithmic bytes
 * (value_bytes + 4) * nnz + 7 * vector_bytes * rows.  Needs a built hierarchy (run a step). */
int shakti_time_amg_smoother(shakti_model* m, int level, int reps, double* ms_per_launch, int64_t* rows,
                             int64_t* nnz, int32_t* value_bytes, int32_t* vector_bytes);
/* One launch of a SELL kernel of AMG level `level`'s part of the V-cycle, launched as the cycle launches it and
 * timed the same way.  `which`: 0 = smoothing step (as shakti_time_amg_smoother), 1 = residual r = b - A x,
 * 2 = restriction onto level + 1 (with that level's first Chebyshev step where the cycle fuses the two),
 * 3 = prolongation x += P x_coarse.  info = {rows, columns, stored entries, longest row, bytes per stored value}
 * of the kernel's matrix (A, R or P), then bytes per vector entry and 1 if the restriction is the fused one.
 * SHAKTI_ERR_INVALID for a kernel the cycle does not run on this rank. */
int shakti_time_amg_level_kernel(shakti_model* m, int level, int which, int reps, double* ms_per_launch, int64_t info[7]);
/* Algorithmic bytes per launch of kernel `which` (SURVEY.md §8d formulas). */
int shakti_kernel_bytes(shakti_model* m, int which, double* bytes);

/* ---------------------------------------------------------------- AMG test hooks
 * What the preconditioner computes, level by level, for a comparison with a float64 reference (tests/amg_reference.py).
 * One rank only (SHAKTI_ERR_INVALID on several); rows and columns are in the model's internal order, which
 * shakti_get_owned maps to caller ids.  They add no work to the solver's own calls.
 * shakti_amg_refresh: rebuilds the preconditioner from the last assembled Jacobian -- full = 1: the whole hierarchy's
 *   numbers (the first call also builds the hierarchy); full = 0: only the fine smoother (diagonal and Chebyshev
 *   bound), the rest stays lagged, as a Newton solve between two scheduled refreshes does.
 * shakti_amg_level_info: info[18] = {rows, columns, n_coarse (0 on the last level), stored entries and longest row of
 *   A, of P, of R (0 on the last level), last, dense coarsest solve (last level only), A runs on its half-precision
 *   copy, the restriction onto this level takes its first Chebyshev step, the cycle's first and last fine sweeps
 *   are fused with its entry and exit (same on every level), number of levels, fp32 cycle, AP and RAP of this level
 *   ran the table-driven SpGEMM}.
 * shakti_amg_get_matrix: `which` 0 = A (level 0: the fine Jacobian), 1 = P, 2 = R, 3 = the fp32 copy of A the cycle
 *   reads, 4 = the fp16 copy of D^-1 A; as CSR (sorted columns), values widened to double.  Call with NULL arrays to
 *   query nnz (rowptr holds rows + 1 entries).
 * shakti_amg_get_vectors: level's dinv (rows doubles) in fp64 and in the cycle's precision, its Chebyshev bound of
 *   lambda_max(D^-1 A) and coefficient table ({1/theta, -, then (c1, c2) of sweep k at 2 + 2k}, *stride doubles;
 *   stride 0 without the Chebyshev smoother).  Any pointer may be NULL.
 * shakti_amg_apply: z = M^-1 r (n_owned doubles each), one V-cycle through the path a Krylov iteration takes. */
int shakti_amg_refresh(shakti_model* m, int full);
int shakti_amg_level_info(shakti_model* m, int level, int64_t info[18]);
int shakti_amg_get_matrix(shakti_model* m, int level, int which, int32_t* rowptr, int32_t* col, double* val, int64_t* nnz);
int shakti_amg_get_vectors(shakti_model* m, int level, double* dinv, double* dinv_cycle, double* lmax, double* coef,
                           int32_t* stride);
int shakti_amg_apply(shakti_model* m, const double* r, double* z);

/* ---------------------------------------------------------------- multi-GPU
 * One process per GPU.  Rank 0 calls shakti_comm_unique_id, the 128-byte id is broadcast by
 * the host program (torch.distributed), then every rank calls shakti_comm_init BEFORE
 * shakti_create.  Replaces MPI.COMM_WORLD (main.py:11) and the DOLFINx/PETSc scatters. */
int shakti_comm_unique_id(uint8_t id[128]);
int shakti_comm_init(const uint8_t id[128], int rank, int nranks, int device);
int shakti_comm_finalize(void);
/* Owned vertices of this rank in caller numbering, in the rank's internal order (the order
 * of the gathers of solvers.py:205-208).  Query the count with ids == NULL. */
int shakti_get_owned(shakti_model* m, int32_t* ids, int64_t* n_owned);

/* ---------------------------------------------------------------- host-side helpers
 * Pure host code (no CUDA device needed): the one-time preprocessing that replaces DOLFINx'
 * dofmap / sparsity-pattern / partitioning work, exposed so it can be checked on its own. */
int shakti_host_csr_pattern(int64_t n_vert, int64_t n_cell, const int32_t* cells, int32_t* rowptr,
                            int32_t* col, int64_t* nnz);
int shakti_host_locate_dirichlet(int64_t n_vert, int64_t n_cell, const int32_t* cells,
                                 const uint8_t* marker, int32_t* dofs, int64_t cap, int64_t* n_out);
/* The rank-local mesh the device code works on (what shakti_create builds for `rank` of
 * `nranks`): internal ordering, owned + ghost vertices, owner-computes cell overlap, SELL
 * pattern, scatter table, winning cells, halo maps. */
typedef struct shakti_host_mesh shakti_host_mesh;
int shakti_host_mesh_create(int64_t n_vert, int64_t n_cell, const double* xy, const int32_t* cells,
                            int rank, int nranks, int reorder, shakti_host_mesh** out);
int shakti_host_mesh_destroy(shakti_host_mesh* hm);
typedef enum shakti_host_array {
  SHAKTI_HM_L2G = 0,        /* n_local: local vertex -> caller id (owned first)          */
  SHAKTI_HM_CELLS = 1,      /* 3*n_cell_local: local vertex ids                          */
  SHAKTI_HM_CELL_L2G = 2,   /* n_cell_local: caller cell ids                             */
  SHAKTI_HM_ROWPTR = 3,     /* n_owned+1: CSR of owned rows (local column ids)           */
  SHAKTI_HM_COL = 4,        /* nnz_local                                                 */
  SHAKTI_HM_SLICE_PTR = 5,  /* n_slices+1: SELL-32 entry offsets                         */
  SHAKTI_HM_SELL_COL = 6,   /* padded entries                                            */
  SHAKTI_HM_SLOT = 7,       /* 9*n_cell_local, k-major: SELL position of (cell,a,b) or -1 */
  SHAKTI_HM_DIAG_POS = 8,   /* n_owned                                                   */
  SHAKTI_HM_WIN = 9,        /* 4*n_owned: winning cell's local vertex ids + local index  */
  SHAKTI_HM_WIN_CELL = 10,  /* n_owned: winning cell, caller cell id                     */
  SHAKTI_HM_NBR_RANK = 11,  /* n_nbrs                                                    */
  SHAKTI_HM_NBR_SEND_PTR = 12, /* n_nbrs+1 offsets into SEND_IDX                         */
  SHAKTI_HM_NBR_SEND_IDX = 13, /* owned local ids to send, concatenated per neighbour    */
  SHAKTI_HM_NBR_RECV = 14,  /* 2*n_nbrs: (first ghost local id, count) per neighbour     */
  /* row-block plan of the atomics-free assembly kernel (csrc/prep.h AssemblyBlocks) */
  SHAKTI_HM_AB_INFO = 15,   /* rows_per_block, n_blocks, max_cells, max_verts, ok         */
  SHAKTI_HM_AB_EPTR = 16,   /* n_blocks+1                                                 */
  SHAKTI_HM_AB_ELEMS = 17,  /* local cell ids per block                                   */
  SHAKTI_HM_AB_LV = 18,     /* 3 per block cell: block-local vertex index                 */
  SHAKTI_HM_AB_HPTR = 19,   /* n_blocks+1                                                 */
  SHAKTI_HM_AB_HALO = 20,   /* halo vertices per block (local ids)                        */
  SHAKTI_HM_AB_INCPTR = 21, /* n_owned+1                                                  */
  SHAKTI_HM_AB_INC = 22,    /* (cell index in block)*4 + local vertex index               */
  SHAKTI_HM_AB_SRC = 23,    /* per padded SELL entry: two 16-bit gather codes (as int32 bits) */
  SHAKTI_HM_CELL_COUNTED = 24 /* n_cell_local: 1 on exactly one rank per cell (the owner of its vertex with the
                                 smallest caller id), else 0: the cells whose integrals this rank contributes */
} shakti_host_array;
/* Size query (out == NULL) or copy of one of the arrays above. */
int shakti_host_mesh_array(shakti_host_mesh* hm, int which, int32_t* out, int64_t* n);
/* Strength-of-connection filter (|a_ij| >= theta sqrt(|a_ii a_jj|), theta <= 0: all connections) and greedy
 * aggregation of a square CSR matrix, as the AMG set-up does on each level; agg_out[i] in [0, *n_agg) or -1. */
int shakti_host_amg_aggregate(int32_t n, const int32_t* rowptr, const int32_t* col, const double* val, double theta,
                              const uint8_t* exclude, int32_t* agg_out, int32_t* n_agg);
/* Host-only self test of the symmetric-heap allocator behind the multi-GPU staging buffers (csrc/comm.cu): a
 * deterministic sequence of `rounds` allocations / releases on a heap of heap_bytes; *violations counts
 * misaligned or overlapping blocks, accepted double frees and a heap that does not coalesce back to one block. */
int shakti_host_heap_selftest(int64_t heap_bytes, int32_t rounds, int32_t* violations);
/* info[0..5] = n_owned, n_local, n_cell_local, nnz_local, padded SELL entries, n_nbrs */
int shakti_host_mesh_info(shakti_host_mesh* hm, int64_t info[6]);

#ifdef __cplusplus
}
#endif
#endif /* SHAKTI_B200_H */
