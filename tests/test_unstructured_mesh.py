"""Unstructured test meshes on the CPU (no GPU needed): the assembly plan state each mesh of tests/unstructured.py is
built to reach, that the per-row F / J distances of the GPU tests see an error confined to the smallest cells, the
water-budget identity of the CPU reference on a graded mesh, and that factoring the fields out of make_case into
case_on left every existing case unchanged."""
import hashlib

import numpy as np
import pytest

import unstructured as U
from common import case_on, make_case, make_oracle, relinf
from unstructured import TOL_ROW_F, TOL_ROW_J, f_row_scale, row_dist_F, row_dist_J

DT = 3600.0


@pytest.fixture(scope="module")
def meshes():
    return {n: U.mesh(n) for n in ("U0", "U64", "U32", "UA")}


@pytest.mark.parametrize("name,reorder", list(U.PLAN))
def test_plan_state(meshes, name, reorder):
    """128-, 64- and 32-row assembly blocks and the refused plan (atomic fallback), chosen from the mesh's shape."""
    xy, cells = meshes[name]
    assert U.plan_state(xy, cells, reorder) == U.PLAN[name, reorder]


def test_hubs_sit_inside_and_outside_the_storage_disc(meshes):
    for name in ("U64", "U32", "UA"):
        xy, cells = meshes[name]
        f = case_on(xy, cells)[2]
        hubs = U.MESHES[name][2]
        for (cx, cy, _, K), inside in zip(hubs, (True, False)):
            v = int(np.argmin(np.hypot(xy[:, 0] - cx, xy[:, 1] - cy)))
            assert np.count_nonzero(cells == v) == K
            assert (f["storage"][v] == 1.0) == inside


# make_case's arrays before case_on was factored out of it.  z_b (cos * sin) is left out: numpy's vectorised cos/sin
# may round differently on other CPUs; every other array is exactly rounded arithmetic on seeded draws.
MAKE_CASE_DIGEST = "7a225c8c3cf40b0423849069cdeddb4bdb062efdc2168fc01b34bcffdb21a7bb"
MAKE_CASE_CALLS = [dict(seed=s) for s in range(33)] + [
    dict(nx=40, ny=28, seed=11), dict(nx=48, ny=32, seed=23), dict(nx=20, ny=14, seed=3), dict(nx=32, ny=24, seed=1),
    dict(seed=4, neg_b=True, turbulent=False), dict(seed=6, storage=False), dict(scramble=False, diagonal="right")]


def _digest(calls):
    d = hashlib.sha256()
    for kw in calls:
        xy, cells, f, bc, N_bdry = make_case(**kw)
        for a in (xy, cells, bc, np.float64(N_bdry)) + tuple(f[k] for k in sorted(f) if k != "z_b"):
            d.update(np.ascontiguousarray(a).tobytes())
    return d.hexdigest()


def test_make_case_unchanged():
    assert _digest(MAKE_CASE_CALLS) == MAKE_CASE_DIGEST
    xy, _, f, _, _ = make_case(seed=9)
    assert np.array_equal(f["z_b"], 50 * np.cos(xy[:, 0] / 2e4) * np.sin(xy[:, 1] / 1.5e4))


def test_per_row_metric_sees_small_cells(meshes):
    """Kbar of the ten smallest cells scaled by (1 + 1e-9) in the oracle: the per-row distances of the GPU tests see
    it, the global relative norm (max |dJ| / max |J|) does not."""
    xy, cells = meshes["U0"]
    o = make_oracle(*case_on(xy, cells, seed=0))
    Fo, Jo = o.assemble(DT)
    small = np.argsort(o.detabs)[:10]
    kb = o.kbar()[small]
    gpgp = np.einsum("eak,ebk->eab", o.gradphi[small], o.gradphi[small])
    plain = o.element_FJ

    def mutated(dt, N=None, want_J=True):
        # cell e's diffusion terms: Kbar_e grad h . grad phi_a in F, -Kbar_e / (rho_w g) grad phi_a . grad phi_b in J
        Fe, Je = plain(dt, N, want_J)
        gh = o._cell_grad(o.head(o.N if N is None else N))[small]
        Fe = Fe.copy()
        Fe[small] += 1e-9 * kb[:, None] * np.einsum("ek,eak->ea", gh, o.gradphi[small])
        if Je is not None:
            Je = Je.copy()
            Je[small] -= 1e-9 * (kb / (o.p.rho_w * o.p.g))[:, None, None] * gpgp
        return Fe, Je

    o.element_FJ = mutated
    Fm, Jm = o.assemble(DT)
    dJ, dF = row_dist_J(Jm, Jo, o.rowptr), row_dist_F(Fm, Fo, f_row_scale(o, DT))
    print(f"MUTATION small-cell Kbar: J per row {dJ:.3e}, F per row {dF:.3e}, "
          f"J global {relinf(Jm, Jo):.3e}, F global {relinf(Fm, Fo):.3e}")
    assert dJ > 10 * TOL_ROW_J and dF > 10 * TOL_ROW_F
    assert relinf(Jm, Jo) < 1e-12 and relinf(Fm, Fo) < 1e-12


def test_budget_identity_of_the_reference(meshes):
    """outflow = input - cm melt + closure + storage + imbalance for the CPU record on a graded mesh."""
    from budget_reference import oracle_diagnostics
    xy, cells = meshes["U0"]
    o = make_oracle(*case_on(xy, cells, seed=1))
    o.N = o.N_n * (1 + 0.01 * np.sin(xy[:, 0] / 3e3))
    r = oracle_diagnostics(o, DT)
    cm = 1 / o.p.rho_i - 1 / o.p.rho_w
    scale = abs(r["input"]) + cm * abs(r["melt"]) + abs(r["closure"]) + abs(r["storage"]) + abs(r["outflow"])
    rhs = r["input"] - cm * r["melt"] + r["closure"] + r["storage"] + r["imbalance"]
    assert abs(r["outflow"] - rhs) <= 1e-12 * scale, r
    assert r["storage"] != 0 and r["outflow"] != 0 and r["area"] == pytest.approx(5e9, rel=1e-12)
