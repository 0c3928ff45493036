"""Water-budget diagnostics without a GPU: the cell-counting rule behind the multi-rank sums, and the discrete
identity  outflow = input - cm melt + closure + storage + imbalance  on the CPU oracle."""
import numpy as np
import pytest

from common import make_case, make_oracle
from budget_reference import oracle_diagnostics
from oracle.shakti_oracle import ShaktiOracle, dirichlet_dofs
from shakti_b200 import capi, meshgen

DT = 3600.0


def _ragged_mesh():
    """Jittered, scrambled rectangle with 40 % of the cells dropped and the orphaned nodes pruned."""
    rng = np.random.default_rng(3)
    xy, cells = meshgen.rectangle(9, 7, 1.0, 1.0, jitter=0.2, seed=2, diagonal="random")
    xy, cells = meshgen.scramble(xy, cells, seed=4)
    keep = rng.random(cells.shape[0]) > 0.4
    keep[0] = True
    cells = cells[keep]
    used = np.zeros(xy.shape[0], bool)
    used[cells.ravel()] = True
    cells = np.ascontiguousarray((np.cumsum(used) - 1)[cells], dtype=np.int32)
    return np.ascontiguousarray(xy[used]), cells


@pytest.mark.parametrize("kind", ["make_case", "ragged"])
@pytest.mark.parametrize("nranks", [1, 2, 3, 8])
def test_every_cell_is_counted_on_exactly_one_rank(kind, nranks):
    if kind == "make_case":
        xy, cells = make_case()[:2]
    else:
        xy, cells = _ragged_mesh()
    count = np.zeros(cells.shape[0], dtype=np.int64)
    for r in range(nranks):
        hm = capi.HostMesh(xy, cells, r, nranks)
        flag, cl2g = hm.array("cell_counted"), hm.array("cell_l2g")
        assert flag.shape == (hm.n_cell,) and set(np.unique(flag)) <= {0, 1}
        np.add.at(count, cl2g[flag == 1], 1)
        # the counting rank owns the cell's vertex with the smallest caller id
        owned = set(hm.array("l2g")[:hm.n_owned].tolist())
        for e, f in zip(cl2g, flag):
            assert (int(cells[e].min()) in owned) == bool(f)
    assert np.all(count == 1)


def _rectangle_oracle():
    """Hand-checkable case: no geothermal flux, no flux, no previous melt, storage off: melt is exactly zero."""
    xy, cells = meshgen.rectangle(20, 10, 100e3, 50e3, jitter=0.2, seed=1, diagonal="random")
    o = ShaktiOracle(xy, cells)
    x, y = xy[:, 0], xy[:, 1]
    o.z_b[:] = 50 * np.cos(x / 2e4) * np.sin(y / 1.5e4)
    o.z_s[:] = 1000 * np.sqrt((x + 5e3) / 105e3)
    o.inputs[:] = 1e-8 * (1 + np.random.default_rng(0).random(o.nv))
    o.b[:] = 2e-3
    o.N_n[:] = 0.37e6
    o.set_dirichlet(dirichlet_dofs(xy, cells, lambda X: np.isclose(X[0], 0.0)), 0.37e6)
    o.start()
    return o


def test_oracle_hand_checkable_rectangle():
    o = _rectangle_oracle()
    d = oracle_diagnostics(o, DT)
    assert d["melt"] == 0.0 and d["storage"] == 0.0
    assert abs(d["area"] - 5e9) <= 1e-14 * 5e9
    assert abs(d["water_volume"] - 2e-3 * d["area"]) <= 1e-14 * 2e-3 * d["area"]
    assert d["N_min"] == d["N_max"] == 0.37e6 and abs(d["N_mean"] - 0.37e6) <= 1e-14 * 0.37e6 and d["b_max"] == 2e-3
    o.newton(DT)
    d = oracle_diagnostics(o, DT)
    assert d["outflow"] > 0
    assert abs(d["outflow"] - (d["input"] + d["closure"] + d["imbalance"])) <= 1e-12 * abs(d["outflow"])


def test_oracle_budget_closes_with_every_term_active():
    o = make_oracle(*make_case(turbulent=True, storage=True))
    cm = 1 / o.p.rho_i - 1 / o.p.rho_w
    for dt in o.dt_schedule(np.linspace(0, 3 * DT, 4))[:3]:
        o.step(dt)
    # the state of a converged solve: the next Newton solve, before the nodal updates
    o.newton(DT)
    d = oracle_diagnostics(o, DT)
    assert all(d[k] != 0 for k in ("input", "melt", "closure", "storage", "outflow"))
    scale = abs(d["input"]) + cm * abs(d["melt"]) + abs(d["closure"]) + abs(d["storage"]) + abs(d["outflow"])
    rhs = d["input"] - cm * d["melt"] + d["closure"] + d["storage"] + d["imbalance"]
    assert abs(d["outflow"] - rhs) <= 1e-10 * scale
    assert abs(d["imbalance"]) <= np.sqrt(o.nv) * d["residual"]


def test_multi_gpu_diagnostics_script_imports_without_gpus():
    """tests/multi_gpu_diagnostics_check.py runs under torchrun on >= 2 GPUs only; it must import anywhere."""
    import importlib
    mod = importlib.import_module("multi_gpu_diagnostics_check")
    assert callable(mod.main)
