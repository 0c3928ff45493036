"""The one-thread-per-row fp32 SELL kernels of the V-cycle (smoother, residual, restriction, prolongation of the AMG
levels of >= 300 000 rows) load a whole row before its gathers when no row of the matrix has more than 8 entries, and
run the plain loop otherwise (sell_row.h).

The row product itself is checked bit for bit by tests/sell_row_check.cu: on random slices of every width 0 ... 8,
the load-before-gather path, the plain loop and a host chain of fmaf in entry order give the same bits.

End to end, C4's grid on 360 000 vertices (rows of 7 entries: the fine level on the load-before-gather path) and
the same grid with fans of 8 triangles spliced in around a few vertices (rows of 9 entries at the fan centres: the
fine level on the plain loop).  On each mesh:

- a linear solve reaches its tolerance in the true residual ||F - J dx||, computed here from the assembled CSR;
- replaying the V-cycle as a CUDA graph gives the same bits and iteration counts as issuing it kernel by kernel;
- two transient steps give the fields of the CPU oracle to 1e-8, with the same Newton iteration counts.  The
  oracle's sparse LU takes about a minute for two steps at this size, so this runs on the grid without fans only
  (the fine level on the load-before-gather path).
"""
import shutil
import subprocess
from pathlib import Path

import numpy as np
import pytest
import scipy.sparse as sp

from common import relinf

pytestmark = pytest.mark.gpu

NSIDE = 600             # 360 000 vertices: the fine level runs the one-thread-per-row kernels
RTOL = 1e-10
CENTRES = ((150, 150), (300, 420), (450, 250), (200, 480))     # grid vertices (ix, iy), away from the boundary
FANS = {0: 8, 1: 0}     # fan size k -> row bound the fine level's fp32 kernels take (0: plain loop)


def fan_case(k):
    """configs.dofs16m(NSIDE) with the 2k x 2k quads around each of CENTRES replaced by a fan of 8k triangles from
    the centre vertex to the patch's boundary ring (k = 0: the grid as is).  The patch's other interior vertices
    are removed and the vertex fields follow the renumbering."""
    from shakti_b200 import configs
    case = configs.dofs16m(nside=NSIDE, nsteps=6)
    if k == 0:
        return case
    n = NSIDE                                 # vertices per grid row; vertex id = iy * n + ix
    xy, cells = case.xy, case.cells
    keep_cell = np.ones(cells.shape[0], bool)
    drop_vert = np.zeros(xy.shape[0], bool)
    fans = []
    for cx, cy in CENTRES:
        inside = (np.abs(cells % n - cx).max(axis=1) <= k) & (np.abs(cells // n - cy).max(axis=1) <= k)
        keep_cell &= ~inside
        gx, gy = np.meshgrid(np.arange(cx - k + 1, cx + k), np.arange(cy - k + 1, cy + k))
        inner = (gy * n + gx).ravel()
        drop_vert[inner[inner != cy * n + cx]] = True
        ring = ([(x, cy - k) for x in range(cx - k, cx + k)] + [(cx + k, y) for y in range(cy - k, cy + k)] +
                [(x, cy + k) for x in range(cx + k, cx - k, -1)] + [(cx - k, y) for y in range(cy + k, cy - k, -1)])
        ring = [y * n + x for x, y in ring]
        fans += [(cy * n + cx, ring[i], ring[(i + 1) % len(ring)]) for i in range(len(ring))]
    cells = np.concatenate([cells[keep_cell], np.asarray(fans, cells.dtype)])
    new_id = np.cumsum(~drop_vert) - 1
    cells = new_id[cells].astype(case.cells.dtype)
    xy = xy[~drop_vert]
    e1, e2 = xy[cells[:, 1]] - xy[cells[:, 0]], xy[cells[:, 2]] - xy[cells[:, 0]]
    assert np.all(e1[:, 0] * e2[:, 1] - e1[:, 1] * e2[:, 0] > 0)     # the fans are oriented like the grid's cells
    case.xy, case.cells = xy, cells
    case.fields = {f: v[~drop_vert] for f, v in case.fields.items()}
    assert not drop_vert[case.bc_dofs].any()
    case.bc_dofs = new_id[case.bc_dofs].astype(case.bc_dofs.dtype)
    return case


ROOT = Path(__file__).resolve().parent.parent


def test_row_product_bitwise(tmp_path):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    exe = tmp_path / "sell_row_check"
    subprocess.run([nvcc, "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a",
                    "-I", str(ROOT / "shakti-fenics_b200" / "csrc"), str(ROOT / "tests" / "sell_row_check.cu"),
                    "-o", str(exe)], check=True, capture_output=True, timeout=300)
    out = subprocess.run([str(exe)], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0 and out.stdout.startswith("ok"), out.stdout[-2000:]


def _longest_row(rowptr):
    return int(np.diff(rowptr).max())


def _bound(width):
    return 8 if width <= 8 else 0


@pytest.fixture(scope="module", params=list(FANS), ids=[f"fan{k}" for k in FANS])
def fan(request):
    from shakti_b200 import capi, configs
    case = fan_case(request.param)
    m = capi.Model(case.xy, case.cells, precond="amg", linear_rtol=RTOL)
    configs.apply_case(m, case)
    m.snapshot()
    yield request.param, case, m
    m.close()


def test_mesh_puts_the_fine_level_in_each_row_bound(fan):
    k, case, m = fan
    rowptr, _ = m.csr()
    assert case.n_vert >= 300000
    assert _bound(_longest_row(rowptr)) == FANS[k]


def test_linear_solve_true_residual_graph_on_off(fan):
    k, case, m = fan
    m.rollback()
    rowptr, col = m.csr()
    F, Jval = m.assemble(3600.0)
    J = sp.csr_matrix((Jval, col, rowptr), shape=(case.n_vert, case.n_vert))
    res = {}
    for graph in (1, 0):
        m.set_options(amg_cuda_graph=graph)
        res[graph] = m.linear_solve(F)[:2]
    levels = m.stats()["amg_levels"]
    m.set_options(amg_cuda_graph=1)       # the next solve rebuilds the hierarchy
    (dx1, it1), (dx0, it0) = res[1], res[0]
    interior = np.ones(case.n_vert, bool)
    interior[case.bc_dofs] = False
    r = (F - J @ dx1)[interior]
    assert np.linalg.norm(r) <= 5 * RTOL * np.linalg.norm(F[interior])
    assert it1 == it0 and np.array_equal(dx1, dx0)
    assert levels >= 3


def test_transient_steps_against_oracle(fan):
    from oracle.shakti_oracle import ShaktiOracle
    k, case, m = fan
    if k != 0:
        pytest.skip("oracle run on the grid without fans only (module docstring)")
    m.rollback()
    o = ShaktiOracle(case.xy, case.cells, backend="c", permc_spec="MMD_AT_PLUS_A")
    for f in ("z_b", "z_s", "G", "inputs", "storage", "b", "N_n", "melt_n"):
        getattr(o, f)[:] = case.fields[f]
    o.q[:] = case.fields["q"]
    o.set_dirichlet(case.bc_dofs, case.N_bdry)
    o.start()
    dts = case.dts(2)
    its_o = [o.step(dt)[0] for dt in dts]
    its_m = [m.step(dt)[0] for dt in dts]
    assert its_m == its_o
    for name, ref in (("N", o.N), ("b", o.b), ("melt_n", o.melt_n)):
        assert relinf(m.get_field(name), ref) < 1e-8, name
    assert relinf(m.get_flux(), o.q) < 1e-8
