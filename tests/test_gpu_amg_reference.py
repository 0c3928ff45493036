"""The AMG hierarchy and V-cycle, level by level, against the float64 scipy reference of tests/amg_reference.py, on
every kernel path of csrc/amg.cu.  The Krylov tests elsewhere only see iteration counts move when the preconditioner
is subtly wrong; these compare what it computes.

Inputs: the Jacobian from Model.assemble, reordered by owned() into the library's internal order, must be bitwise
the exported level-0 operator.  Then, per case:

- bitwise: dinv = 1/diag on every level; R = P^T; the fp32 copies (values and dinv) are the rounded fp64 ones and
  the fp16 copy is f16(f32(dinv_i a_ij)); the first (plain), second (captured) and third (replayed) apply give the
  same z; apply(r1), apply(r2), apply(r1) gives the same z for r1 twice; apply(2 r) = 2 apply(r);
- per entry, each level from the library's own inputs of that level (amg_reference.compare_levels): P within
  TOL_P of its row's largest entry, A_{l+1} within TOL_GALERKIN (|R||A||P|)_ij (the summation-error bound), identical
  patterns, Chebyshev coefficients within TOL_COEF;
- z of the fp64 cycle within TOL_Z64 (relative infinity norm) of the reference cycle, of the fp32 cycle within
  TOL_Z32;
- discrimination: each mutation of the reference (amg_reference.MUTATIONS and prolong_omega 0.66) moves z by at
  least 10 x the tolerance in use, so the tolerance tells a right cycle from a subtly wrong one.

Largest distances measured on a B200, over all cases, next to the bound in use (each bound is at most 100 x its
measured distance; the smallest discrimination ratio seen at that bound is in brackets):
  P                6.6e-16   TOL_P        1e-14
  Galerkin         5.4e-16   TOL_GALERKIN 5e-14
  coefficients     4.2e-16   TOL_COEF     1e-14
  z, fp64 cycle    1.3e-14   TOL_Z64      1e-12   (prolong_omega 0.66 on the small mesh: 7.5e9 x)
  z, dense J^-1    1.8e-15   TOL_Z64
  z, fp32 cycle    3.9e-7    TOL_Z32      3e-5    (prolong_omega 0.66 on the small mesh: 250 x)
  z, fp16 level 0  3.3e-7    TOL_Z32              (5.1e-4 against the reference without the half switch)
The whole file runs in about 50 s on a B200 host; the 3M-row case (test_largest_mesh_table_spgemm) takes 23 s of it.
"""
import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import scipy.sparse as sp

import amg_reference as ar

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent
TOL_P = 1e-14
TOL_GALERKIN = 5e-14
TOL_COEF = 1e-14
TOL_Z64 = 1e-12
TOL_Z32 = 3e-5
LARGE = 300000       # rows from which a level runs the one-thread-per-row kernels (kChebyWideRowsBelow)
TABLE = 400000       # rows above which the numeric SpGEMM runs table-driven (spgemm_numeric)


# ------------------------------------------------------------------------------------------------ plumbing
def fine_system(m, n_vert, bc_dofs):
    """-> (F, J, exclude) in the library's internal order (owned())."""
    rowptr, col = m.csr()
    F, Jval = m.assemble(3600.0)
    J = sp.csr_matrix((Jval, col, rowptr), shape=(n_vert, n_vert))
    own = m.owned()
    Ji = sp.csr_matrix(J[own][:, own])
    Ji.sort_indices()
    isbc = np.zeros(n_vert, bool)
    isbc[bc_dofs] = True
    return F[own], Ji, isbc[own]


def exports(m):
    out = []
    for l in range(m.amg_level_info(0)["levels"]):
        info = m.amg_level_info(l)
        v = m.amg_vectors(l)
        e = dict(info=info, A=m.amg_matrix(l, "A"), dinv=v["dinv"], dinv_cycle=v["dinv_cycle"], last=bool(info["last"]))
        if v["coef"].size:
            e["coef"] = v["coef"]
        if not e["last"]:
            e["P"], e["R"] = m.amg_matrix(l, "P"), m.amg_matrix(l, "R")
        if info["fp32_cycle"]:
            e["low"] = m.amg_matrix(l, "valh" if info["uses_half"] else "valf")
        out.append(e)
    return out


def precision_copies_exact(exp):
    """The cycle's copies are the rounded fp64 values: valf = f32(a), valh = f16(f32(dinv_i a_ij)), dinv_cycle."""
    ok = True
    for e in exp:
        A = e["A"]
        if not e["info"]["fp32_cycle"]:
            ok &= bool(np.array_equal(e["dinv_cycle"], e["dinv"]))
            continue
        ok &= bool(np.array_equal(e["dinv_cycle"], e["dinv"].astype(np.float32).astype(np.float64)))
        rows = np.repeat(np.arange(A.shape[0]), np.diff(A.indptr))
        if e["info"]["uses_half"]:
            want = (e["dinv"][rows] * A.data).astype(np.float32).astype(np.float16).astype(np.float64)
        else:
            want = A.data.astype(np.float32).astype(np.float64)
        ok &= ar.same_csr(e["low"], sp.csr_matrix((want, A.indices, A.indptr), shape=A.shape))
    return ok


def apply_checks(m, r1, r2):
    """Bitwise properties of Model.amg_apply -> z(r1)."""
    z = [m.amg_apply(r1) for _ in range(3)]
    assert np.array_equal(z[0], z[1]) and np.array_equal(z[1], z[2]), "plain / captured / replayed cycles differ"
    z2 = m.amg_apply(r2)
    assert np.array_equal(m.amg_apply(r1), z[0]) and not np.array_equal(z2, z[0]), "state carried between cycles"
    assert np.array_equal(m.amg_apply(2.0 * r1), 2.0 * z[0]), "apply(2r) != 2 apply(r)"
    return z[0]


def check_levels(exp, J, excl, opt, measured):
    assert ar.same_csr(exp[0]["A"], J), "exported level-0 operator is not the reordered assembled Jacobian"
    res = ar.compare_levels([dict(e) for e in exp], excl, opt)
    measured.update({k: max(measured.get(k, 0.0), res[k]) for k in ("P", "galerkin", "coef")})
    assert res["patterns"] and res["dinv_exact"] and res["R_exact"], res
    assert res["P"] <= TOL_P and res["galerkin"] <= TOL_GALERKIN and res["coef"] <= TOL_COEF, res
    assert precision_copies_exact(exp)


def check_z(z, H, r, tol, name, measured, J=None, excl=None):
    zr = ar.vcycle(H, r)
    d = ar.rel_inf(z, zr)
    measured[name] = max(measured.get(name, 0.0), d)
    print(f"MEASURED {name} {d:.3e}")
    assert d <= tol, (name, d)
    if J is not None:
        disc = ar.discrimination(H, r, tol, J, excl)
        print(f"DISCRIMINATION {name} " + " ".join(f"{k}={v:.3g}" for k, v in disc.items()))
        assert min(disc.values()) >= 10, (name, disc)


MEASURED = {}


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    print("MEASURED max " + json.dumps(MEASURED))


# ------------------------------------------------------------------------------------------------ small mesh
def _small(cycle, **opt):
    from common import make_case, make_model
    xy, cells, f, bc, N_bdry = make_case(nx=24, ny=16, seed=3)
    m = make_model(xy, cells, f, bc, N_bdry, amg_fp32_cycle=1 if cycle == "fp32" else 0, **opt)
    F, J, excl = fine_system(m, xy.shape[0], bc)
    return m, F, J, excl


@pytest.mark.parametrize("cycle", ["fp64", "fp32"])
def test_small_hierarchy_warp_kernels(cycle):
    """KG = 8 kernels and the warp SpGEMM on every level of a >= 3-level hierarchy."""
    m, F, J, excl = _small(cycle, amg_coarse_size=16)
    m.amg_refresh(True)
    z = apply_checks(m, F, np.random.default_rng(1).standard_normal(F.size))
    exp = exports(m)
    assert len(exp) >= 3 and all(e["info"]["rows"] < LARGE and not e["info"]["table_AP"] for e in exp)
    opt = ar.Options.of(m.options)
    check_levels(exp, J, excl, opt, MEASURED)
    H = ar.build(J, excl, opt)
    tol = TOL_Z64 if cycle == "fp64" else TOL_Z32
    check_z(z, H, F, tol, f"z_{cycle}", MEASURED, J, excl)
    m.close()


def test_one_level_dense_inverse():
    m, F, J, excl = _small("fp64", amg_max_levels=1)
    m.amg_refresh(True)
    z = apply_checks(m, F, np.random.default_rng(2).standard_normal(F.size))
    exp = exports(m)
    assert len(exp) == 1 and exp[0]["info"]["dense_coarse"] and exp[0]["info"]["rows"] <= ar.DENSE_MAX
    d = ar.rel_inf(z, np.linalg.solve(J.toarray(), F))
    MEASURED["z_dense"] = d
    print(f"MEASURED z_dense {d:.3e}")
    assert d <= TOL_Z64
    m.close()


# ------------------------------------------------------------------------------------------------ large mesh
NSIDE = 600          # 360 000 rows: level 0 on the one-thread-per-row kernels, rows of 7 entries (RB = 8)
CONFIGS = {          # name: options, seams_apply, restrict_starts(level 1), discrimination checks
    "cheby_2_2": (dict(), 1, 1, True),
    "cheby_2_1": (dict(amg_postsmooth=1), 1, 1, False),
    "cheby_1_1": (dict(amg_presmooth=1, amg_postsmooth=1), 0, 0, False),
    "cheby_3_0": (dict(amg_presmooth=3, amg_postsmooth=0), 0, 1, False),
    "cheby_0_3": (dict(amg_presmooth=0, amg_postsmooth=3), 0, 0, False),
    "jacobi": (dict(amg_smoother="jacobi"), 0, 0, False),
    "fp64": (dict(amg_fp32_cycle=0), 0, 1, True),
}
BASE = dict(amg_presmooth=2, amg_postsmooth=2, amg_smoother="chebyshev", amg_fp32_cycle=1, amg_max_levels=12)


def large_case(nside=NSIDE):
    from shakti_b200 import configs
    return configs.dofs16m(nside=nside, nsteps=4)


def large_model(case, **opt):
    from shakti_b200 import capi, configs
    m = capi.Model(case.xy, case.cells, **opt)
    configs.apply_case(m, case)
    m.snapshot()
    return m


@pytest.fixture(scope="module")
def large():
    case = large_case()
    m = large_model(case)
    F, J, excl = fine_system(m, case.n_vert, case.bc_dofs)
    H = ar.build(J, excl, ar.Options.of(m.options))
    yield case, m, F, J, excl, H
    m.close()


@pytest.mark.parametrize("name", list(CONFIGS))
def test_large_mesh_cycle(large, name):
    """Level 0 on KG = 1 with RB = 8 (fp32); the seams and restrict_cheby_first on and off per smoother setting."""
    case, m, F, J, excl, H = large
    cfg, seams, starts, disc = CONFIGS[name]
    m.set_options(**{**BASE, **cfg})
    m.rollback()
    m.assemble(3600.0)
    m.amg_refresh(True)
    z = apply_checks(m, F, np.random.default_rng(3).standard_normal(F.size))
    info = [m.amg_level_info(l) for l in range(m.amg_level_info(0)["levels"])]
    i0 = info[0]
    assert i0["rows"] >= LARGE and i0["A_width"] <= 8 and not i0["uses_half"] and i0["levels"] >= 3
    assert info[1]["rows"] < LARGE
    assert i0["seams_apply"] == seams and info[1]["restrict_starts"] == starts, (name, i0, info[1])
    opt = ar.Options.of(m.options)
    if name in ("cheby_2_2", "fp64"):
        check_levels(exports(m), J, excl, opt, MEASURED)
    else:
        assert precision_copies_exact(exports(m))
    Hc = H.with_options(presmooth=opt.presmooth, postsmooth=opt.postsmooth, smoother=opt.smoother)
    fp32 = m.options.amg_fp32_cycle == 1
    check_z(z, Hc, F, TOL_Z32 if fp32 else TOL_Z64, "z_fp32" if fp32 else "z_fp64", MEASURED,
            J if disc else None, excl)


def test_large_mesh_chebyshev_coarsest(large):
    """Two levels: the coarsest level (> 1024 rows) is smoothed by 8 Chebyshev sweeps instead of a dense solve."""
    case, m, F, J, excl, _ = large
    m.set_options(**{**BASE, "amg_max_levels": 2})
    m.rollback()
    m.assemble(3600.0)
    m.amg_refresh(True)
    z = apply_checks(m, F, np.random.default_rng(4).standard_normal(F.size))
    i1 = m.amg_level_info(1)
    assert i1["levels"] == 2 and i1["last"] and not i1["dense_coarse"] and i1["rows"] > ar.DENSE_MAX
    opt = ar.Options.of(m.options)
    H = ar.build(J, excl, opt)
    assert H.levels[1].last and H.levels[1].inverse is None
    check_z(z, H, F, TOL_Z32, "z_fp32", MEASURED)


@pytest.mark.parametrize("cycle", ["fp32", "fp64"])
def test_large_mesh_lagged_hierarchy(large, cycle):
    """Full refresh, then N changes, J is re-assembled and only the fine smoother is refreshed (one-pass refresh in
    the fp32 cycle, dinv + Gershgorin kernels in the fp64 one): level 0 on the new J, the rest on the old."""
    case, m, F, J, excl, H = large
    m.set_options(**{**BASE, "amg_fp32_cycle": 1 if cycle == "fp32" else 0})
    m.rollback()
    m.assemble(3600.0)
    m.amg_refresh(True)
    coarse = m.amg_matrix(1, "A")
    N = case.fields["N_n"] * (1.0 + 0.05 * np.sin(case.xy[:, 0] / 7e3))
    m.set_field("N", N)
    F2, J2, _ = fine_system(m, case.n_vert, case.bc_dofs)
    assert not ar.same_csr(J2, J)
    m.amg_refresh(False)
    z = m.amg_apply(F2)
    exp = exports(m)
    assert ar.same_csr(exp[0]["A"], J2) and ar.same_csr(exp[1]["A"], coarse)
    assert np.array_equal(exp[0]["dinv"], ar.dinv_of(J2)) and precision_copies_exact(exp)
    opt = ar.Options.of(m.options)
    ref = ar.cheby_coef(ar.gershgorin(J2, exp[0]["dinv"]), opt.ratio, opt.coef_sweeps)
    assert np.max(np.abs(exp[0]["coef"] - ref)) <= TOL_COEF * np.max(np.abs(ref))
    tol = TOL_Z32 if cycle == "fp32" else TOL_Z64
    check_z(z, H.with_fine(J2), F2, tol, f"z_{cycle}", MEASURED)
    # the lagged reference is not the fresh one: the check sees which hierarchy the cycle used
    assert ar.rel_inf(z, ar.vcycle(ar.build(J2, excl, opt), F2)) >= 10 * tol
    m.rollback()


def test_large_mesh_plain_row_loop():
    """Fans of 8 triangles give rows of 9 entries: level 0's fp32 kernels take the plain loop (RB = 0)."""
    from test_gpu_sell_kernels import fan_case
    case = fan_case(8)
    m = large_model(case)
    F, J, excl = fine_system(m, case.n_vert, case.bc_dofs)
    m.amg_refresh(True)
    z = apply_checks(m, F, np.random.default_rng(5).standard_normal(F.size))
    i0 = m.amg_level_info(0)
    assert i0["rows"] >= LARGE and i0["A_width"] > 8 and i0["fp32_cycle"] and i0["seams_apply"]
    assert precision_copies_exact(exports(m))
    check_z(z, ar.build(J, excl, ar.Options.of(m.options)), F, TOL_Z32, "z_fp32", MEASURED)
    m.close()


def test_largest_mesh_table_spgemm():
    """Level 0 and level 1 above 400 000 rows: AP and RAP of both run the table-driven SpGEMM, level 1 the
    one-thread-per-row smoother."""
    case = large_case(1750)
    m = large_model(case)
    F, J, excl = fine_system(m, case.n_vert, case.bc_dofs)
    m.amg_refresh(True)
    z = m.amg_apply(F)
    info = [m.amg_level_info(l) for l in range(m.amg_level_info(0)["levels"])]
    assert info[0]["rows"] > TABLE and info[1]["rows"] > TABLE, [i["rows"] for i in info]
    assert info[0]["table_AP"] and info[0]["table_RAP"] and info[1]["table_AP"], info[:2]
    exp = exports(m)
    opt = ar.Options.of(m.options)
    check_levels(exp, J, excl, opt, MEASURED)
    check_z(z, ar.build(J, excl, opt), F, TOL_Z32, "z_fp32", MEASURED)
    m.close()


_FP16_CHILD = r"""
import json, sys
import numpy as np
sys.path[:0] = [sys.argv[1], sys.argv[1] + "/shakti-fenics_b200", sys.argv[1] + "/tests"]
import amg_reference as ar
from test_gpu_amg_reference import apply_checks, exports, fine_system, large_case, large_model, precision_copies_exact
case = large_case()
m = large_model(case)
F, J, excl = fine_system(m, case.n_vert, case.bc_dofs)
m.amg_refresh(True)
z = apply_checks(m, F, np.random.default_rng(6).standard_normal(F.size))
exp = exports(m)
half = [l for l, e in enumerate(exp) if e["info"]["uses_half"]]
H = ar.build(J, excl, ar.Options.of(m.options))
print(json.dumps(dict(half=half, seams=exp[0]["info"]["seams_apply"], copies=precision_copies_exact(exp),
                      d=ar.rel_inf(z, ar.vcycle(H.with_half(half), F)), d_plain=ar.rel_inf(z, ar.vcycle(H, F)))))
"""


def test_large_mesh_half_precision_copy():
    """SHAKTI_AMG_FP16=1 (read once per process, so in a child): level 0 runs on f16(f32(D^-1 A)), without seams."""
    env = dict(os.environ, SHAKTI_AMG_FP16="1")
    out = subprocess.run([sys.executable, "-c", _FP16_CHILD, str(ROOT)], env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-3000:]
    res = json.loads(out.stdout.strip().splitlines()[-1])
    print(f"MEASURED z_fp16 {res['d']:.3e} (against the reference without the half switch: {res['d_plain']:.3e})")
    MEASURED["z_fp16"] = res["d"]
    assert res["half"] == [0] and res["seams"] == 0 and res["copies"], res
    assert res["d"] <= TOL_Z32, res
