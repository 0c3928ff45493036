"""Moulins on the CPU: the hydrograph lookup of the reference, the reference's residual, Jacobian and water budget
with moulins, and the snapping of md.moulins in solvers (model construction replaced by a fake, no GPU)."""
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
for p in (ROOT / "shakti-fenics_b200" / "source", ROOT / "shakti-fenics_b200" / "setups"):
    if str(p) not in sys.path:
        sys.path.insert(0, str(p))

from budget_reference import oracle_diagnostics  # noqa: E402
from common import make_case  # noqa: E402
from moulin_reference import MoulinOracle, hydrograph, moulin_diagnostics  # noqa: E402

DT = 3600.0
CM = 1 / 917 - 1 / 1000


def direct(tk, qk, t, period=0.0):
    """Q(t) written out knot interval by knot interval."""
    if period > 0:
        t = tk[0] + (t - tk[0]) - period * np.floor((t - tk[0]) / period)
    if t <= tk[0]:
        return qk[0]
    if t >= tk[-1]:
        return qk[-1]
    j = np.searchsorted(tk, t, side="right") - 1
    return qk[j] + (qk[j + 1] - qk[j]) * (t - tk[j]) / (tk[j + 1] - tk[j])


def test_hydrograph_lookup():
    tk = np.array([0.0, 3600.0, 7200.0, 20000.0, 86400.0])
    qk = np.array([1.0, 3.0, 0.0, 0.5, 1.0])
    for t, want in ((0.0, 1.0), (3600.0, 3.0), (7200.0, 0.0), (86400.0, 1.0),      # knots
                    (1800.0, 2.0), (5400.0, 1.5),                                   # between knots
                    (-50.0, 1.0), (-1e9, 1.0), (9e4, 1.0), (1e12, 1.0)):           # outside the range
        assert hydrograph(tk, qk, t) == want, t
    ts = np.linspace(-3e5, 3e5, 2001)
    got = hydrograph(tk, qk, ts)
    assert np.allclose(got, [direct(tk, qk, t) for t in ts], rtol=1e-15, atol=1e-15)
    # period: t and t + k * period give the same Q, and Q is the direct formula of the wrapped time
    per = 86400.0
    got = hydrograph(tk, qk, ts, period=per)
    assert np.allclose(got, [direct(tk, qk, t, per) for t in ts], rtol=1e-14, atol=1e-14)
    assert np.allclose(hydrograph(tk, qk, ts + 3 * per, period=per), got, rtol=1e-12, atol=1e-12)
    assert hydrograph(tk, qk, per + 1800.0, period=per) == pytest.approx(2.0, rel=1e-15)
    assert hydrograph(tk, qk, -per + 5400.0, period=per) == pytest.approx(1.5, rel=1e-15)
    # a period longer than the table: constant after the last knot until the wrap
    assert hydrograph(tk[:3], qk[:3], 2e4 + 1e5, period=1e5) == 0.0


def _moulin_oracle(seed=0):
    xy, cells, f, bc, N_bdry = make_case(seed=seed)
    o = MoulinOracle(xy, cells)
    for k in ("z_b", "z_s", "G", "inputs", "storage", "b", "N_n", "melt_n"):
        getattr(o, k)[:] = f[k]
    o.q[:] = f["q"]
    o.set_dirichlet(bc, N_bdry)
    o.start()
    rng = np.random.default_rng(seed)
    free = np.setdiff1d(np.arange(o.nv), bc)
    v = rng.choice(free, size=6, replace=False)
    v = np.concatenate([v, v[:2]])                            # two vertices carry two moulins each
    tk = np.linspace(0.0, 86400.0, 25)
    mo = [(int(a), tk, q * (1.0 + 0.5 * np.sin(2 * np.pi * tk / 86400.0))) for a, q in zip(v, rng.uniform(0.5, 3, v.size))]
    o.set_moulins(mo, period=86400.0)
    return o, bc


def test_reference_residual_changes_by_minus_q_and_jacobian_is_unchanged():
    o, bc = _moulin_oracle()
    o.t = 5000.0
    F1, J1 = o.assemble(DT)
    mo = o.moulins
    o.moulins = []
    F0, J0 = o.assemble(DT)
    o.moulins = mo
    q = o.moulin_discharge(o.t + DT)
    want = np.zeros(o.nv)
    for (v, _, _), qk in zip(mo, q):
        want[v] -= qk
    rows = np.unique([v for v, _, _ in mo])
    assert rows.size == len(mo) - 2 and not np.isin(rows, bc).any()
    assert np.array_equal(F1 - F0 == 0, want == 0)
    assert np.allclose((F1 - F0)[rows], want[rows], rtol=1e-12, atol=0)
    assert np.array_equal(J1, J0)


def test_reference_budget_identity_with_moulins():
    """After a converged solve the record with moulins closes (outflow = input - cm melt + closure + storage +
    imbalance), its input is int inputs + sum Q, and the imbalance (moulin rows included) is a Newton remainder."""
    o, bc = _moulin_oracle(seed=3)
    o.t = 2 * 3600.0
    it, conv = o.newton(DT)
    assert conv and it >= 1
    d = moulin_diagnostics(o, DT)
    plain = oracle_diagnostics(o, DT)
    qsum = o.moulin_discharge(o.t + DT).sum()
    assert qsum > 0 and d["input"] == plain["input"] + qsum
    scale = abs(d["input"]) + CM * abs(d["melt"]) + abs(d["closure"]) + abs(d["storage"]) + abs(d["outflow"])
    rhs = d["input"] - CM * d["melt"] + d["closure"] + d["storage"] + d["imbalance"]
    assert abs(d["outflow"] - rhs) <= 1e-10 * scale
    F, _ = o.assemble(DT, want_J=False)
    isbc = np.zeros(o.nv, dtype=bool)
    isbc[bc] = True
    assert abs(d["imbalance"] - F[~isbc].sum()) <= 1e-10 * scale
    # a Newton remainder (bounded by the residual norm); without the moulin rows it would be about +sum Q
    assert abs(d["imbalance"]) <= np.sqrt(o.nv) * d["residual"] + 1e-12 * scale and abs(d["imbalance"]) < 1e-3 * qsum


def _md(tmp_path, moulins):
    from _synthetic import md_from_case
    from shakti_b200 import configs, fem
    case = configs.moulins_like(nx=20, ny=4, n_moulins=5, nsteps=4)
    md = md_from_case(fem.comm_world(), case, str(ROOT / "shakti-fenics_b200" / "setups" / "setup_moulins_like.py"),
                      results_name=str(tmp_path / "out"))
    md.moulins = moulins
    md.moulin_period = 86400.0
    return md, case


class _FakeModel:
    made = []

    def __init__(self, xy, cells, params=None, device=-1, **opts):
        self.calls = []
        _FakeModel.made.append(self)

    def __getattr__(self, name):
        return lambda *a, **kw: self.calls.append((name, a, kw))


def test_solvers_snaps_moulins_and_refuses_outflow_dofs(tmp_path, monkeypatch):
    import solvers
    from shakti_b200.fem import Function
    monkeypatch.setattr(solvers.capi, "Model", _FakeModel)
    tk, qk = np.array([0.0, 43200.0, 86400.0]), np.array([1.0, 2.0, 1.0])

    def build(moulins):
        md, case = _md(tmp_path, moulins)
        N, N_n, b, melt_n = (Function(md.V) for _ in range(4))
        q = Function(md.V_flux)
        solvers.pde_solver(md, N, N_n, b, q, melt_n, md.lake_bdry, solvers.Constant(md.domain, 360.0))
        return md, case, _FakeModel.made[-1]

    md, case, _ = build([])
    xy0 = case.xy
    # targets: slightly off three interior vertices, and one moulin given by vertex id
    targets = [int(np.argmin(np.hypot(xy0[:, 0] - x, xy0[:, 1] - y))) for x, y in ((31e3, 9e3), (55e3, 12e3), (80e3, 3e3))]
    moulins = [(xy0[v, 0] + 7.0, xy0[v, 1] - 5.0, tk, qk) for v in targets] + [(targets[0], tk, 2 * qk)]
    md, case, fake = build(moulins)
    names = [c[0] for c in fake.calls]
    assert names.index("set_dirichlet") < names.index("set_moulins")
    _, (vertex, times, discharges), kw = fake.calls[names.index("set_moulins")]
    assert vertex.tolist() == targets + [targets[0]] and kw == dict(period=86400.0)
    assert np.array_equal(times[0], tk) and np.array_equal(discharges[3], 2 * qk)
    # a moulin next to the outflow edge x = 0 snaps onto a Dirichlet dof: an error that names it
    bc = case.bc_dofs
    with pytest.raises(ValueError, match=r"moulin 1 at .* snapped to vertex %d .*outflow" % bc[2]):
        build([moulins[0], (xy0[bc[2], 0] + 10.0, xy0[bc[2], 1], tk, qk)])
    with pytest.raises(ValueError, match="moulin 0 at vertex %d .*outflow" % bc[0]):
        build([(int(bc[0]), tk, qk)])
