"""Unstructured test meshes (test infrastructure; scipy stays out of shakti_b200/): graded, jittered Delaunay
triangulations of the 100 km x 50 km domain of tests/common.py, optionally with fans of K triangles spliced in around
single vertices ("hubs").  Vertex valences of 5-10 and more, ragged rows and graded cell sizes reach the code paths
that the structured rectangles never do: the 64- and 32-row assembly blocks, the refused assembly plan (atomic
fallback), wide SELL slices and the searching SpGEMM of the large AMG levels.

Every builder asserts the properties its tests rely on (longest row, valence >= 10 somewhere, min/max cell-area
ratio, aspect ratio of the cells away from the hubs, no zero-area cell), so a change of scipy's triangulation cannot
quietly weaken a test."""
import functools

import numpy as np
from scipy.spatial import Delaunay

from oracle.shakti_oracle import csr_pattern
from shakti_b200 import meshgen

LX, LY = 100e3, 50e3
STORAGE_HUB = (50e3, 25e3)        # inside the storage disc of common.case_on (radius 15 km around the centre)
OUTER_HUB = (80e3, 12e3)          # outside it


def _triangulate(pts):
    """Delaunay triangulation without hull slivers or unreferenced points -> (xy, cells)."""
    cells = Delaunay(pts).simplices.astype(np.int64)
    X = pts[cells]
    d1, d2 = X[:, 1] - X[:, 0], X[:, 2] - X[:, 0]
    det = np.abs(d1[:, 0] * d2[:, 1] - d2[:, 0] * d1[:, 1])
    cells = cells[det > 1e-9 * det.max()]
    used = np.zeros(len(pts), bool)
    used[cells.ravel()] = True
    remap = np.cumsum(used) - 1
    return np.ascontiguousarray(pts[used]), np.ascontiguousarray(remap[cells], dtype=np.int32)


def graded_delaunay(nx, ny, seed=0, grade=1.6, drop=0.2, jitter=0.3):
    """Staggered lattice of (nx+1) x (ny+1) points, interior points jittered by +-jitter cells and a seeded fraction
    `drop` of them removed, x graded as LX * s**grade (the smallest cells on the Dirichlet edge x = 0) -> points."""
    rng = np.random.default_rng(seed)
    s, t = np.meshgrid(np.linspace(0, 1, nx + 1), np.linspace(0, 1, ny + 1))
    s = s + 0.5 * (np.arange(ny + 1)[:, None] % 2) / nx
    s[:, 0] = 0.0                 # staggered rows start on the edge too (no sliver cells along x = 0)
    inner = (s > 0) & (s < 1) & (t > 0) & (t < 1)
    s = s + inner * rng.uniform(-jitter, jitter, s.shape) / nx
    t = t + inner * rng.uniform(-jitter, jitter, t.shape) / ny
    keep = ~inner | (rng.random(s.shape) > drop)
    s, t = np.clip(s[keep], 0, 1), t[keep]
    return np.unique(np.c_[LX * s ** grade, LY * t], axis=0)


def add_fans(pts, hubs):
    """For each hub (cx, cy, radius, K): drop the points within 1.3 radius, add the centre and a ring of K points on
    the circle.  The Delaunay triangulation then has a fan of K triangles around the centre (row width K + 1)."""
    pts = np.asarray(pts, dtype=np.float64)
    for cx, cy, R, K in hubs:
        pts = pts[np.hypot(pts[:, 0] - cx, pts[:, 1] - cy) > 1.3 * R]
        a = 2 * np.pi * np.arange(K) / K
        pts = np.concatenate([pts, [[cx, cy]], np.c_[cx + R * np.cos(a), cy + R * np.sin(a)]])
    return pts


def mesh_stats(xy, cells, hubs=()):
    """-> dict(n_vert, n_cell, row_max, valence_max, area_ratio, aspect_max (cells away from the hubs), area_min)."""
    rp, _ = csr_pattern(xy.shape[0], cells)
    w = np.diff(rp)
    X = xy[cells]
    d1, d2, d3 = X[:, 1] - X[:, 0], X[:, 2] - X[:, 0], X[:, 2] - X[:, 1]
    area = 0.5 * np.abs(d1[:, 0] * d2[:, 1] - d2[:, 0] * d1[:, 1])
    L2 = np.max(np.stack([np.einsum("ij,ij->i", d, d) for d in (d1, d2, d3)], 1), axis=1)
    away = np.ones(cells.shape[0], bool)
    cen = X.mean(axis=1)
    for cx, cy, R, _ in hubs:
        away &= np.hypot(cen[:, 0] - cx, cen[:, 1] - cy) > 2.0 * R
    return dict(n_vert=int(xy.shape[0]), n_cell=int(cells.shape[0]), row_max=int(w.max()), valence_max=int(w.max() - 1),
                n_valence10=int((w >= 11).sum()), area_ratio=float(area.max() / area.min()),
                aspect_max=float((L2 / area)[away].max()), area_min=float(area.min()))


def build(nx, ny, hubs=(), seed=0, grade=1.6):
    """Graded Delaunay mesh with fans at `hubs`, scrambled (random numbering, both cell orientations) and checked:
    longest row K_max + 1 (or <= 16 without hubs), some vertex of valence >= 10, graded cell areas (ratio >= 20),
    cells away from the hubs of bounded aspect ratio, no zero-area cell -> (xy, cells)."""
    pts = add_fans(graded_delaunay(nx, ny, seed=seed, grade=grade), hubs)
    xy, cells = _triangulate(pts)
    xy, cells = meshgen.scramble(xy, cells, seed=seed + 5)
    st = mesh_stats(xy, cells, hubs)
    kmax = max((K for *_, K in hubs), default=0)
    if hubs:
        assert st["row_max"] == kmax + 1, st
    else:
        assert 11 <= st["row_max"] <= 16, st
    assert st["n_valence10"] > 0, st
    assert st["area_ratio"] >= 20.0, st
    assert st["aspect_max"] <= 100.0, st
    assert st["area_min"] > 0.0, st
    return xy, cells


# name: (nx, ny, hubs, grade).  U0 has about 12 000 vertices; the hub sizes are chosen so that the assembly plan takes the
# asserted path (tests/test_unstructured_mesh.py: 128-, 64- and 32-row blocks, refused).  UL is above the 400 000-row
# threshold of the table-driven SpGEMM and its hub gives A.P a row wider than the table's 96 entries; its grading is
# milder so that its 1040 columns keep the cells along x = 0 within the aspect-ratio bound.
MESHES = {
    "U0": (170, 85, (), 1.6),
    "U64": (170, 85, ((*STORAGE_HUB, 4e3, 200), (*OUTER_HUB, 3e3, 120)), 1.6),
    "U32": (170, 85, ((*STORAGE_HUB, 4e3, 320), (*OUTER_HUB, 3e3, 120)), 1.6),
    "UA": (170, 85, ((*STORAGE_HUB, 4e3, 500), (*OUTER_HUB, 3e3, 120)), 1.6),
    "UL": (1040, 520, ((*STORAGE_HUB, 1e3, 480),), 1.3),
}
# (mesh, reorder): rows per assembly block and ok of HostMesh.ab_info, one rank.  In the caller's (scrambled) order a
# block of rows touches more cells, so the plan shrinks its blocks or is refused one hub size earlier.
PLAN = {("U0", 1): (128, 1), ("U64", 1): (64, 1), ("U32", 1): (32, 1), ("UA", 1): (None, 0),
        ("U0", 0): (64, 1), ("U64", 0): (32, 1), ("U32", 0): (None, 0), ("UA", 0): (None, 0)}


def plan_state(xy, cells, reorder=1, rank=0, nranks=1):
    """-> (rows per block or None when the plan is refused, ok) of the library's assembly plan for this mesh."""
    from shakti_b200 import capi
    rb, _, _, _, ok = (int(v) for v in capi.HostMesh(xy, cells, rank, nranks, reorder).array("ab_info"))
    return (rb if ok else None), ok


@functools.lru_cache(maxsize=None)
def mesh(name):
    """The mesh `name` of MESHES, built once per process (callers must not modify the arrays)."""
    nx, ny, hubs, grade = MESHES[name]
    return build(nx, ny, hubs, grade=grade)


# ---------------------------------------------------------------------------------------------- per-row distances
# On a graded mesh the largest rows dominate a global relative norm, so F and J are compared row by row.
TOL_ROW_J = 1e-13
TOL_ROW_F = 1e-11       # F carries the rounding of grad h (differences of ~1 km heads) over the smallest cells


def row_dist_J(J, Jo, rowptr):
    """max_i ||J_i - Jo_i||_inf / ||Jo_i||_inf over the rows of a CSR pattern."""
    d = np.maximum.reduceat(np.abs(J - Jo), rowptr[:-1])
    s = np.maximum.reduceat(np.abs(Jo), rowptr[:-1])
    return float(np.max(d / s))


def f_row_scale(o, dt):
    """Summation-error scale of each row of the oracle's assembled F: sum over the row's cells of |element residual|
    and |Dirichlet lifting|, or |F_i| on a Dirichlet row.  A row whose terms cancel is compared with its terms, not
    with what is left of them."""
    Fe, Je = o.element_FJ(dt)
    c = o.cells
    isbc = np.zeros(o.nv, dtype=bool)
    isbc[o.bc_dofs] = True
    gx = np.where(isbc[c], o.N_bdry - o.N[c], 0.0)
    s = np.zeros(o.nv)
    np.add.at(s, c.ravel(), (np.abs(Fe) + np.abs(np.einsum("eab,eb->ea", Je, gx))).ravel())
    Fo, _ = o.assemble(dt, want_J=False)
    s[isbc] = np.abs(Fo[isbc])
    return np.maximum(s, 1e-300)


def row_dist_F(F, Fo, scale):
    """max_i |F_i - Fo_i| / scale_i (scale: f_row_scale)."""
    return float(np.max(np.abs(F - Fo) / scale))
