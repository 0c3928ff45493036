"""The CUDA path on unstructured meshes (tests/unstructured.py) against the CPU oracle: graded Delaunay meshes with
valences of 5-10 and fans of up to 500 triangles, in the library's Morton order and in the caller's scrambled order.
Each test asserts which path it reaches (HostMesh.ab_info for the assembly plan, amg_level_info for the SpGEMM):

- U0 / U64 / U32 / UA: the assembly plan with 128-, 64- and 32-row blocks and the refused plan (cell atomics + the
  Dirichlet pass); CSR pattern and winning cells bit-exact, Kbar, F and J (with and without J), a second plan assembly
  bitwise equal, SpMV, the nodal updates with the b clamp, the water-budget record, transient runs (AMG / Jacobi);
- U32: the AMG hierarchy and V-cycle level by level (test_gpu_amg_reference.py's checks and mutations);
- UL (> 400 000 vertices, one fan of 480): level 0 above both size thresholds of csrc/amg.cu with an A.P row wider
  than the 96 entries of the table-driven SpGEMM, so the searching SpGEMM builds A.P; every Galerkin level, F and J
  against the oracle's C backend, the one-thread-per-row SpMV per row, and a linear solve checked through its true
  residual.

F and J are compared PER ROW (max_i ||dJ_i||_inf / ||Jo_i||_inf, and the same for F with a floor): on a graded mesh the
largest rows dominate a global relative norm, which would miss an error confined to the smallest cells.
test_unstructured_mesh.py:test_per_row_metric_sees_small_cells shows the difference with a mutation of the oracle.

Largest distances measured on a B200, next to the bound in use.  Each bound is at most 100 x its measured distance;
where a bound shared with the structured-mesh tests is wider (the water-budget record's 1e-12), a tighter one of this
file is asserted as well:
  Kbar (relative inf norm)          5.4e-16   5e-14
  J per row                         1.8e-15   TOL_ROW_J   1e-13  (small-cell Kbar mutation: 4.9e-10)
  F per row, scaled by its terms    1.4e-12   TOL_ROW_F   1e-11  (small-cell Kbar mutation: 3.2e-10)
  J / F per row on UL, C backend    1.5e-15 / 1.2e-11   TOL_ROW_J / TOL_ROW_F_C 1e-10
  SpMV per row, by sum |a_ij x_j|   1.7e-15 (KG = 8), 5.2e-16 (UL, one thread per row)   1e-14
  q / melt_n / b updates            7.6e-14 / 5.0e-14 / 9.4e-16   1e-13 / 1e-13 / 5e-14 (b_min clamp count equal)
  water-budget record               3.7e-16   3e-14 (and test_gpu_diagnostics.py's 1e-12)
  transient N / b / melt_n / q      4.0e-10 / 3.6e-9 / 4.3e-11 / 7.4e-10   TRANSIENT, Newton counts equal
  AMG on U32: P, Galerkin, coef     1.4e-15, 5.3e-16, 6.6e-16 (TOL_P 1e-14, TOL_GALERKIN 5e-14, TOL_COEF 1e-14)
  AMG on U32: z fp64 / fp32 cycle   3.0e-15 / 2.7e-7   TOL_Z64_U 2e-13 / TOL_Z32_U 2.5e-5, every mutation moves z
                                    by >= 260 x the bound
  UL: P, Galerkin, coef             1.4e-15, 6.2e-16, 6.6e-16 (largest over three runs); A.P row 158 wide, table_AP 0
  UL: linear solve                  8.7e-11 true residual over the non-Dirichlet rows, relative to the right-hand side
                                    the solve sees (linear_rtol 1e-10)   TOL_SOLVE x linear_rtol = 1e-9
The whole file runs in about 40 s on a B200 host.
"""
import json

import numpy as np
import pytest
import scipy.sparse as sp

import amg_reference as ar
import unstructured as U
from common import case_on, make_model, make_oracle, relinf
from unstructured import TOL_ROW_F, TOL_ROW_J, f_row_scale, row_dist_F, row_dist_J
from test_gpu_amg_reference import apply_checks, check_levels, check_z, exports, fine_system

pytestmark = pytest.mark.gpu

DT = 3600.0
TOL_Z64_U = 2e-13       # V-cycle z on U32 against the reference, fp64 cycle (relative inf norm)
TOL_Z32_U = 2.5e-5      # and fp32 cycle
TRANSIENT = dict(N=1e-8, b=1e-8, N_n=1e-8, melt_n=4e-9, q=1e-8)      # fields after six steps, relative inf norm
TOL_ROW_F_C = 1e-10     # F against the oracle's C backend, which orders its operations differently
TOL_SOLVE = 10          # true interior residual of a linear solve, in units of its linear_rtol
WIDE_ROWS = 300000      # rows from which the fp64 SpMV runs one thread per row (kWideRowsBelow)
TABLE = 400000          # rows above which the numeric SpGEMM is table-driven (spgemm_numeric)
TABLE_WIDTH = 96        # widest C row the table-driven SpGEMM holds in shared memory (build_spgemm_plan)

MEASURED = {}


def _measure(name, d):
    MEASURED[name] = max(MEASURED.get(name, 0.0), float(d))
    print(f"MEASURED {name} {d:.3e}")
    return d


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    print("MEASURED max " + json.dumps(MEASURED))


MESHES = ["U0", "U64", "U32", "UA"]
mesh = U.mesh


@pytest.fixture(scope="module", params=[(n, r) for n in MESHES for r in (1, 0)], ids=[f"{n}-{'morton' if r else 'caller'}" for n in MESHES for r in (1, 0)])
def case(request):
    name, reorder = request.param
    xy, cells = mesh(name)
    assert U.plan_state(xy, cells, reorder) == U.PLAN[name, reorder]
    c = case_on(xy, cells, seed=0)
    o = make_oracle(*c)
    m = make_model(*c, reorder=reorder)
    yield name, reorder, c, o, m
    m.close()


def test_pattern_winning_cells_kbar(case):
    _, _, _, o, m = case
    rowptr, col = m.csr()
    assert np.array_equal(rowptr, o.rowptr) and np.array_equal(col, o.col)
    assert np.array_equal(m.winning_cells(), o.win_cell)
    assert _measure("kbar", relinf(m.kbar(), o.kbar())) < 5e-14


def test_residual_and_jacobian_per_row(case):
    name, reorder, _, o, m = case
    F, J = m.assemble(DT)
    Fo, Jo = o.assemble(DT)
    dJ, dF = row_dist_J(J, Jo, o.rowptr), row_dist_F(F, Fo, f_row_scale(o, DT))
    _measure("J_row", dJ)
    _measure("F_row", dF)
    assert dJ <= TOL_ROW_J and dF <= TOL_ROW_F, (name, reorder, dJ, dF)
    F1, none = m.assemble(DT, want_J=False)
    assert none is None
    _measure("F_row", row_dist_F(F1, Fo, f_row_scale(o, DT)))
    assert row_dist_F(F1, Fo, f_row_scale(o, DT)) <= TOL_ROW_F
    if U.PLAN[name, reorder][1]:                  # the row-block plan uses no atomics: bitwise reproducible
        F2, J2 = m.assemble(DT)
        assert np.array_equal(F, F2) and np.array_equal(J, J2)


def test_spmv_per_row(case):
    _, _, _, o, m = case
    m.assemble(DT)
    _, Jo = o.assemble(DT)
    A = o.jacobian_matrix(Jo)
    x = np.random.default_rng(3).standard_normal(o.nv)
    y = m.spmv(x)
    ref = A @ x
    scale = abs(A) @ np.abs(x)                    # per row: sum_j |a_ij x_j|, the summation-error scale
    d = float(np.max(np.abs(y - ref) / scale))
    _measure("spmv_row", d)
    assert d <= 1e-14


def test_nodal_updates_with_clamp(case):
    _, reorder, (xy, cells, *_), _, _ = case
    c = case_on(xy, cells, seed=4, neg_b=True, turbulent=False)
    o = make_oracle(*c)
    m = make_model(*c, reorder=reorder)
    try:
        N = c[2]["N_n"] * (1 + 0.01 * np.random.default_rng(5).standard_normal(o.nv))
        o.N = N.copy()
        m.set_field("N", N)
        o.update_q(); m.update_q()
        assert _measure("q", relinf(m.get_flux(), o.q)) < 1e-13
        o.update_melt(); m.update_melt()
        assert _measure("melt_n", relinf(m.get_field("melt_n"), o.melt_n)) < 1e-13
        o.update_b(DT); m.update_b(DT)
        bg = m.get_field("b")
        assert (bg == o.b_min).sum() == (o.b == o.b_min).sum() > 0
        assert _measure("b", relinf(bg, o.b)) < 5e-14
    finally:
        m.close()


def test_water_budget_record(case):
    from budget_reference import oracle_diagnostics
    from test_gpu_diagnostics import _assert_records_close
    from multi_gpu_diagnostics_check import record_errors
    _, _, _, o, m = case
    got, ref = m.diagnostics(DT), oracle_diagnostics(o, DT)
    d = max(v for k, v in record_errors(got, ref, 1 / 917 - 1 / 1000).items() if k not in ("N_min", "N_max", "b_max"))
    _measure("budget", d)
    _assert_records_close(got, ref)                   # the structured-mesh bounds (1e-12; minima and maxima equal)
    assert d <= 3e-14


@pytest.mark.parametrize("name,pc", [("U0", "amg"), ("U32", "amg"), ("UA", "jacobi")])
def test_transient_run(name, pc):
    xy, cells = mesh(name)
    c = case_on(xy, cells, seed=2)
    o = make_oracle(*c)
    m = make_model(*c, precond=pc, linear_max_it=5000)
    try:
        dts = o.dt_schedule(np.linspace(0, 8 * DT, 9))[:6]
        its_o = [o.step(dt)[0] for dt in dts]
        its_m = list(m.run(dts))
        assert its_m == its_o
        for k, got, ref in (("N", m.get_field("N"), o.N), ("b", m.get_field("b"), o.b), ("N_n", m.get_field("N_n"), o.N_n),
                            ("melt_n", m.get_field("melt_n"), o.melt_n), ("q", m.get_flux(), o.q)):
            d = _measure(f"transient_{k}", relinf(got, ref))
            assert d < TRANSIENT[k], (k, d)
    finally:
        m.close()


@pytest.mark.parametrize("cycle", ["fp64", "fp32"])
def test_amg_levels_on_fan_mesh(cycle):
    """U32: the hierarchy and V-cycle of a mesh with 321-wide rows against the float64 reference, with the mutations
    of amg_reference each moving z by at least 10 x the tolerance."""
    xy, cells = mesh("U32")
    c = case_on(xy, cells, seed=3)
    m = make_model(*c, amg_fp32_cycle=1 if cycle == "fp32" else 0)
    try:
        F, J, excl = fine_system(m, xy.shape[0], c[3])
        m.amg_refresh(True)
        z = apply_checks(m, F, np.random.default_rng(1).standard_normal(F.size))
        exp = exports(m)
        assert len(exp) >= 2 and exp[0]["info"]["A_width"] == 321
        opt = ar.Options.of(m.options)
        check_levels(exp, J, excl, opt, MEASURED)
        check_z(z, ar.build(J, excl, opt), F, TOL_Z64_U if cycle == "fp64" else TOL_Z32_U, f"z_{cycle}", MEASURED, J, excl)
    finally:
        m.close()


# ------------------------------------------------------------------------------------------------ UL
@pytest.fixture(scope="module")
def large():
    xy, cells = U.mesh("UL")
    c = case_on(xy, cells, seed=0)
    m = make_model(*c)
    yield c, m
    m.close()


def test_large_searching_spgemm_and_galerkin(large):
    c, m = large
    F, J, excl = fine_system(m, c[0].shape[0], c[3])
    m.amg_refresh(True)
    i0 = m.amg_level_info(0)
    assert i0["rows"] > TABLE and i0["A_width"] == 481 and not i0["last"]
    A, P = m.amg_matrix(0, "A"), m.amg_matrix(0, "P")
    ap_width = int(np.diff((ar.ones(A) @ ar.ones(P)).indptr).max())
    print(f"UL: level 0 rows {i0['rows']}, A width {i0['A_width']}, A.P width {ap_width}, P width {i0['P_width']}")
    assert ap_width > TABLE_WIDTH
    assert i0["table_AP"] == 0                        # the table refused A.P: the searching SpGEMM built it
    # every level, level 1's Galerkin product (built from the searched A.P) included, within the bounds of
    # test_gpu_amg_reference.py
    check_levels(exports(m), J, excl, ar.Options.of(m.options), MEASURED)
    print("MEASURED UL levels " + json.dumps({k: MEASURED[k] for k in ("P", "galerkin", "coef")}))


def test_large_assembly_and_linear_solve(large):
    c, m = large
    o = make_oracle(*c, backend="c")
    F, J = m.assemble(DT)
    Fo, Jo = o.assemble(DT)
    rowptr, col = m.csr()
    assert np.array_equal(rowptr, o.rowptr) and np.array_equal(col, o.col)
    dJ, dF = row_dist_J(J, Jo, o.rowptr), row_dist_F(F, Fo, f_row_scale(o, DT))
    _measure("UL_J_row", dJ)
    _measure("UL_F_row", dF)
    assert dJ <= TOL_ROW_J and dF <= TOL_ROW_F_C
    # the solve sees F with its Dirichlet rows zeroed (and sets dx = F there): its true residual over the other rows,
    # relative to that right-hand side, must be within a small factor of the tolerance
    rtol = 1e-10
    m.set_options(linear_rtol=rtol, linear_max_it=2000)
    dx, its, relres = m.linear_solve(F)
    A = sp.csr_matrix((J, col, rowptr), shape=(o.nv, o.nv))
    inner = np.ones(o.nv, dtype=bool)
    inner[c[3]] = False
    true = float(np.linalg.norm((F - A @ dx)[inner]) / np.linalg.norm(F[inner]))
    print(f"UL linear solve: {its} iterations, reported {relres:.3e}, true interior residual {_measure('UL_solve', true):.3e}")
    assert np.array_equal(dx[~inner], F[~inner])
    assert relres <= rtol and true <= TOL_SOLVE * rtol


def test_large_spmv_per_row(large):
    """434 000 rows (above kWideRowsBelow, kernels.cu) with a 481-wide row: the one-thread-per-row SpMV, per row
    against scipy on the model's own assembled J."""
    c, m = large
    F, J = m.assemble(DT)
    rowptr, col = m.csr()
    assert m.stats()["n_owned"] >= WIDE_ROWS and np.diff(rowptr).max() == 481
    A = sp.csr_matrix((J, col, rowptr), shape=(F.size, F.size))
    x = np.random.default_rng(4).standard_normal(F.size)
    d = float(np.max(np.abs(m.spmv(x) - A @ x) / (abs(A) @ np.abs(x))))
    _measure("UL_spmv_row", d)
    assert d <= 1e-14
