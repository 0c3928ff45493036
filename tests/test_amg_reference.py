"""CPU tests of the float64 AMG reference (tests/amg_reference.py), each against an independent statement of what it
computes, so that the GPU comparisons in test_gpu_amg_reference.py rest on a checked reference."""
import importlib.util
from dataclasses import replace
from pathlib import Path

import numpy as np
import pytest
import scipy.sparse as sp

import amg_reference as ar
from common import make_case, make_oracle

ROOT = Path(__file__).resolve().parent.parent


def _prototype(n=14):
    spec = importlib.util.spec_from_file_location("amg_prototype", ROOT / "tools" / "amg_prototype.py")
    proto = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(proto)
    A, excl = proto.operator(*proto.mesh(n))
    A.sort_indices()
    return A, excl


def _jacobian():
    """J of a tiny make_case, assembled by the CPU oracle, and its Dirichlet rows."""
    xy, cells, f, bc, N_bdry = make_case(nx=24, ny=16, seed=4)
    o = make_oracle(xy, cells, f, bc, N_bdry)
    _, val = o.assemble(3600.0)
    J = sp.csr_matrix((val, o.col, o.rowptr), shape=(o.nv, o.nv))
    J.sort_indices()
    excl = np.zeros(o.nv, bool)
    excl[bc] = True
    return J, excl


def test_prolongator_equals_dense_construction():
    A, excl = _prototype()
    agg, na = ar.aggregates(A, 0, excl, 0.08)
    P = ar.prolongator(A, ar.dinv_of(A), agg, na, 0.67)
    n = A.shape[0]
    Ad = A.toarray()
    T = np.zeros((n, na))
    T[np.nonzero(agg >= 0)[0], agg[agg >= 0]] = 1.0
    Pd = np.diag((agg >= 0).astype(float)) @ (np.eye(n) - 0.67 * np.diag(1.0 / np.diag(Ad)) @ Ad) @ T
    assert np.abs(P.toarray() - Pd).max() <= 1e-15 * np.abs(Pd).max()
    # the pattern: every (i, agg(j)) of a stored a_ij of a kept row, no more
    S = (np.diag((agg >= 0).astype(float)) @ ((Ad != 0) | np.eye(n, dtype=bool)) @ T) != 0
    assert np.array_equal(P.toarray() != 0, S & (Pd != 0)) and np.array_equal(ar.ones(P).toarray() != 0, S)
    assert (P.getnnz(axis=1)[excl] == 0).all()


def test_one_level_dense_cycle_is_the_inverse():
    J, excl = _jacobian()
    H = ar.build(J, excl, ar.Options(max_levels=1))
    assert len(H.levels) == 1 and H.levels[0].inverse is not None
    b = np.random.default_rng(1).standard_normal(J.shape[0])
    x = np.linalg.solve(J.toarray(), b)
    assert ar.rel_inf(ar.vcycle(H, b), x) < 1e-12


@pytest.mark.parametrize("smoother", ["chebyshev", "jacobi"])
def test_two_level_cycle_without_smoothing_is_the_coarse_correction(smoother):
    A, excl = _prototype()
    H = ar.build(A, excl, ar.Options(max_levels=2, coarse_size=16, presmooth=0, postsmooth=0, smoother=smoother))
    assert len(H.levels) == 2 and H.levels[1].inverse is not None
    L = H.levels[0]
    P, R = L.P.toarray(), L.R.toarray()
    assert np.array_equal(R, P.T)
    b = np.random.default_rng(2).standard_normal(A.shape[0])
    z = P @ np.linalg.solve(R @ A.toarray() @ P, R @ b)
    assert ar.rel_inf(ar.vcycle(H, b), z) < 1e-12


@pytest.mark.parametrize("sweeps", range(1, 9))
def test_chebyshev_coefficients_minimise_the_error_polynomial(sweeps):
    """On D^-1 A = diag(lambda), lambda in [lmax/ratio, lmax], k sweeps from a zero guess leave the error
    p_k(lambda) e with max |p_k| = 1/T_k(theta/delta): the recurrence against the mathematics of Chebyshev
    acceleration, not against a transcription of itself."""
    lmax, ratio = 3.7, 5.0
    lo = lmax / ratio
    theta, delta = (lmax + lo) / 2, (lmax - lo) / 2
    extrema = theta - delta * np.cos(np.arange(sweeps + 1) * np.pi / sweeps)      # where |p_k| is largest
    lam = np.sort(np.concatenate([np.linspace(lo, lmax, 2001), extrema]))
    A = sp.diags(lam).tocsr()
    opt = ar.Options(presmooth=sweeps, max_levels=1)
    L = ar.Level(A, np.ones(lam.size), ar.cheby_coef(lmax, ratio, opt.coef_sweeps + 1), last=False)
    H = ar.Hierarchy([L], opt)
    e = np.ones(lam.size)
    x = ar._smooth(H, 0, A @ e, None, sweeps, ())[0]
    err = e - x
    bound = 1.0 / np.cosh(sweeps * np.arccosh(theta / delta))
    assert abs(np.abs(err).max() - bound) <= 1e-12
    assert np.all(np.abs(err) <= bound * (1 + 1e-12))
    # equioscillation: the extrema reach the bound with alternating signs
    pe = err[np.searchsorted(lam, extrema)]
    assert np.allclose(np.abs(pe), bound, rtol=1e-10, atol=0) and np.all(np.sign(pe[1:]) == -np.sign(pe[:-1]))


def test_non_finite_bound_gives_two():
    for bad in (0.0, -1.0, np.inf, np.nan):
        assert np.array_equal(ar.cheby_coef(bad, 5.0, 8), ar.cheby_coef(2.0, 5.0, 8))


def test_comparison_plumbing_on_the_reference_itself():
    """The comparison functions of the GPU test, fed the reference's own exports: every distance 0, every flag
    true; a relative perturbation of the largest entry of a coarse operator (1e-10) or of P (1e-12) is seen."""
    J, excl = _jacobian()
    opt = ar.Options(coarse_size=16)
    H = ar.build(J, excl, opt)
    assert len(H.levels) >= 3
    exp = ar.exports_of(H)
    res = ar.compare_levels(exp, excl, opt)
    assert res == dict(P=0.0, galerkin=0.0, coef=0.0, patterns=True, dinv_exact=True, R_exact=True)
    bad = [dict(e) for e in exp]
    A2 = bad[2]["A"].copy()
    A2.data[np.argmax(np.abs(A2.data))] *= 1 + 1e-10
    bad[2]["A"] = A2
    assert ar.compare_levels(bad, excl, opt)["galerkin"] > 1e-13
    bad = [dict(e) for e in exp]
    P0 = bad[0]["P"].copy()
    P0.data[np.argmax(np.abs(P0.data))] *= 1 + 1e-12
    bad[0]["P"] = P0
    r = ar.compare_levels(bad, excl, opt)
    assert r["P"] > 1e-14 and not r["R_exact"]


def test_mutations_move_the_cycle():
    """Every mutation of the discrimination checks changes z of a three-level cycle."""
    J, excl = _jacobian()
    H = ar.build(J, excl, ar.Options(coarse_size=16))
    b = np.random.default_rng(3).standard_normal(J.shape[0])
    d = ar.discrimination(H, b, 1e-6, J, excl)
    assert set(d) == set(ar.MUTATIONS) | {"omega"} and min(d.values()) >= 10, d


def test_lagged_and_half_switches():
    J, excl = _jacobian()
    H = ar.build(J, excl, ar.Options(coarse_size=16))
    J2 = J.copy()
    J2.data *= 1.0 + 0.1 * np.cos(np.arange(J2.nnz))
    HL = H.with_fine(J2)
    assert HL.levels[0].A is not H.levels[0].A and HL.levels[1] is H.levels[1]
    assert np.array_equal(HL.levels[0].dinv, ar.dinv_of(J2))
    HH = H.with_half([0])
    rel = abs(HH.levels[0].A - H.levels[0].A).max() / abs(H.levels[0].A).max()
    assert 0 < rel < 1e-3
    b = np.random.default_rng(4).standard_normal(J.shape[0])
    assert 0 < ar.rel_inf(ar.vcycle(HH, b), ar.vcycle(H, b)) < 1e-2


def test_jacobi_cycle_matches_the_prototype():
    """The damped-Jacobi V-cycle against tools/amg_prototype.py's (independent code) on a hierarchy built here."""
    spec = importlib.util.spec_from_file_location("amg_prototype", ROOT / "tools" / "amg_prototype.py")
    proto = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(proto)
    A, excl = _prototype()
    H = ar.build(A, excl, ar.Options(coarse_size=16, smoother="jacobi", max_levels=3))
    H.levels[-1].inverse = np.linalg.inv(H.levels[-1].A.toarray())
    lev = [dict(A=L.A, D=L.A.diagonal(), P=L.P, R=L.R, last=L.last) for L in H.levels]
    b = np.random.default_rng(5).standard_normal(A.shape[0])
    assert ar.rel_inf(ar.vcycle(H, b), proto.vcycle(lev, 0, b, "jacobi", 2)) < 1e-12
    Hc = replace(H, opt=replace(H.opt, smoother="chebyshev"))
    Hc.levels = [replace(L, coef=ar.smoother_coef(L.A, L.dinv, Hc.opt)) for L in H.levels]
    assert ar.rel_inf(ar.vcycle(Hc, b), proto.vcycle(lev, 0, b, "cheb", 2)) < 1e-12
