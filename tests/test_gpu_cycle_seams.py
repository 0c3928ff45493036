"""The AMG preconditioner's per-solve smoother refresh and its Chebyshev coefficients live on the device: a refresh of
the fine smoother changes no kernel argument, so the captured V-cycle is replayed without re-capture.  These tests
run every AMG configuration on a mesh large enough that levels 0 and 1 both use the one-thread-per-row kernels
(level 1 above 300 000 rows), and check that

- a linear solve reaches its tolerance in the true residual ||F - J dx||, computed here from the assembled CSR;
- replaying the cycle as a CUDA graph gives the same bits and iteration counts as issuing it kernel by kernel;
- transient steps, which alternate full refreshes and per-solve smoother refreshes, give the same fields either way.
"""
import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import scipy.sparse as sp

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent
RTOL = 1e-10
CONFIGS = {
    "default": {},
    "fp64_cycle": dict(amg_fp32_cycle=0),
    "jacobi": dict(amg_smoother="jacobi"),
    "sweeps_1_1": dict(amg_presmooth=1, amg_postsmooth=1),
    "sweeps_3_3": dict(amg_presmooth=3, amg_postsmooth=3),
    "sweeps_0_3": dict(amg_presmooth=0, amg_postsmooth=3),
    "sweeps_3_0": dict(amg_presmooth=3, amg_postsmooth=0),
    "one_level": dict(amg_max_levels=1),
    "bicgstab": dict(linear_solver="bicgstab"),
}


def _case():
    from shakti_b200 import configs
    return configs.dofs16m(nside=1450, nsteps=8)      # C4's fields on 2.1M vertices


def _model(case, **opt):
    from shakti_b200 import capi, configs
    m = capi.Model(case.xy, case.cells, **opt)
    configs.apply_case(m, case)
    m.snapshot()
    return m


@pytest.fixture(scope="module")
def sys_():
    case = _case()
    m = _model(case, linear_rtol=RTOL)
    rowptr, col = m.csr()
    F, Jval = m.assemble(3600.0)
    J = sp.csr_matrix((Jval, col, rowptr), shape=(case.n_vert, case.n_vert))
    yield case, m, F, J
    m.close()


def _configure(m, graph, cfg):
    m.set_options(**{**dict(amg_presmooth=2, amg_postsmooth=2, amg_smoother=1, amg_fp32_cycle=1, amg_max_levels=12,
                            linear_solver="gmres"), **cfg, "amg_cuda_graph": graph})


def _solve(m, F, graph, cfg):
    _configure(m, graph, cfg)
    return m.linear_solve(F)


@pytest.mark.parametrize("name", list(CONFIGS))
def test_linear_solve_graph_on_off(sys_, name):
    case, m, F, J = sys_
    cfg = CONFIGS[name]
    m.rollback()
    m.assemble(3600.0)      # the state F and J were taken from
    dx1, it1, _ = _solve(m, F, 1, cfg)
    dx0, it0, _ = _solve(m, F, 0, cfg)
    interior = np.ones(case.n_vert, bool)
    interior[case.bc_dofs] = False
    r = (F - J @ dx1)[interior]
    assert np.linalg.norm(r) <= 5 * RTOL * np.linalg.norm(F[interior]), name
    assert it1 == it0 and np.array_equal(dx1, dx0), name
    if name == "default":
        st = m.stats()
        assert st["amg_levels"] >= 3


def _steps(case, m, graph, cfg, n=4):
    """n steps from the model's snapshot; changing the AMG options rebuilds the hierarchy at the first solve"""
    m.rollback()
    _configure(m, graph, cfg)
    st0 = m.stats()
    its = [m.step(dt)[0] for dt in case.dts(n)]
    out = [m.get_field(f) for f in ("N", "b", "melt_n")] + [m.get_flux()]
    st = m.stats()
    return its, st["linear_its"] - st0["linear_its"], st["amg_refreshes"] - st0["amg_refreshes"], out


@pytest.mark.parametrize("name", ["default", "fp64_cycle", "sweeps_3_3"])
def test_transient_steps_graph_on_off(sys_, name):
    case, m = sys_[:2]
    a = _steps(case, m, 1, CONFIGS[name])
    b = _steps(case, m, 0, CONFIGS[name])
    assert a[0] == b[0] and a[1] == b[1]
    # the default refresh interval leaves solves on a lagged hierarchy (the per-solve smoother refresh)
    assert sum(a[0]) > a[2]
    assert all(np.array_equal(x, y) for x, y in zip(a[3], b[3]))


_FP16_CHILD = r"""
import json, sys
import numpy as np
sys.path[:0] = [sys.argv[1], sys.argv[1] + "/shakti-fenics_b200", sys.argv[1] + "/tests"]
from test_gpu_cycle_seams import _case, _model, _steps
case = _case()
m = _model(case)
a, b = _steps(case, m, 1, {}), _steps(case, m, 0, {})
print(json.dumps(dict(same=a[0] == b[0] and a[1] == b[1] and all(np.array_equal(x, y) for x, y in zip(a[3], b[3])),
                      its=a[0])))
"""


def test_half_precision_fine_level_graph_on_off():
    """SHAKTI_AMG_FP16=1 (read once per process): the fine level's half-precision copy is made after the one-pass
    refresh, from its diagonal"""
    env = dict(os.environ, SHAKTI_AMG_FP16="1")
    out = subprocess.run([sys.executable, "-c", _FP16_CHILD, str(ROOT)], env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    res = json.loads(out.stdout.strip().splitlines()[-1])
    assert res["same"], res
