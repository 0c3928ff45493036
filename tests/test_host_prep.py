"""Host-side preprocessing of the C-ABI library (no GPU needed): CSR pattern bit-exact against
the oracle, Dirichlet location, internal ordering, SELL layout, scatter table, winning cells,
partition + halo maps."""
import ctypes
import re
from pathlib import Path

import numpy as np
import pytest
import scipy.sparse as sp

import unstructured
from oracle.shakti_oracle import ShaktiOracle, csr_pattern, dirichlet_dofs
from shakti_b200 import capi, meshgen

ROOT = Path(__file__).resolve().parent.parent


def test_library_exports_every_declared_symbol():
    header = (ROOT / "include" / "shakti_b200.h").read_text()
    names = set(re.findall(r"\b(shakti_[a-z0-9_]+)\s*\(", header))
    assert len(names) >= 40
    lib = capi.load()
    missing = [n for n in sorted(names) if not hasattr(lib, n)]
    assert not missing, missing
    assert lib.shakti_version().decode().startswith("shakti_b200")


def test_struct_layouts_match_header():
    o = capi.default_options()
    assert (o.newton_rtol, o.newton_atol, o.newton_max_it) == (1e-9, 1e-10, 50)
    assert o.b_min == 1e-5 and o.reorder == 1 and o.gmres_restart > 0
    # the LAST members: any disagreement about the layout in between would show here
    assert o.linear_forcing == 0.01 and o.amg_replicate_below == 100000
    assert o.newton_relaxation == 1.0 and o.newton_line_search == 0      # the reference's plain Newton step
    hdr = (ROOT / "include" / "shakti_b200.h").read_text()
    body = hdr[hdr.index("typedef struct shakti_options {"):hdr.index("} shakti_options;")]
    names = re.findall(r"\b(?:double|int32_t)\s+([^;]+);", body)
    names = [n.strip() for grp in names for n in grp.split(",")]
    assert names == [f for f, _ in capi.Options._fields_]
    body = hdr[hdr.index("typedef struct shakti_stats {"):hdr.index("} shakti_stats;")]
    names = re.findall(r"\b(?:double|int64_t)\s+([^;]+);", body)
    names = [n.strip() for grp in names for n in grp.split(",")]
    assert names == [f for f, _ in capi.Stats._fields_]
    p = capi.default_params()
    import sys
    sys.path.insert(0, str(ROOT / "shakti-fenics_b200" / "source"))
    import params
    for k in params.NAMES:
        assert getattr(p, k) == float(getattr(params, k))


def test_create_without_gpu_fails_loudly():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    xy, cells = meshgen.rectangle(2, 2, 1.0, 1.0)
    with pytest.raises(capi.ShaktiError) as e:
        capi.Model(xy, cells)
    assert e.value.code in (-2, -3)


@pytest.fixture(scope="module")
def mesh():
    xy, cells = meshgen.rectangle(40, 30, 100e3, 50e3, jitter=0.25, diagonal="random")
    return meshgen.scramble(xy, cells)


def test_csr_pattern_bit_exact(mesh):
    xy, cells = mesh
    rp, col = capi.host_csr_pattern(xy.shape[0], cells)
    rp2, col2 = csr_pattern(xy.shape[0], cells)
    assert rp.dtype == np.int32 and col.dtype == np.int32
    assert np.array_equal(rp, rp2) and np.array_equal(col, col2)


def test_locate_dirichlet(mesh):
    xy, cells = mesh
    d = capi.host_locate_dirichlet(xy.shape[0], cells, np.isclose(xy[:, 0], 0.0))
    assert np.array_equal(d, dirichlet_dofs(xy, cells, lambda X: np.isclose(X[0], 0.0)))
    assert capi.host_locate_dirichlet(xy.shape[0], cells, np.zeros(xy.shape[0], bool)).size == 0


def _sell_to_csr(hm, vals, nv):
    l2g = hm.array("l2g")
    rowptr, lcol = hm.array("rowptr"), hm.array("col")
    sp_, scol = hm.array("slice_ptr"), hm.array("sell_col")
    rows, cols, vv = [], [], []
    for r in range(hm.n_owned):
        base = sp_[r >> 5] + (r & 31)
        for k in range(rowptr[r + 1] - rowptr[r]):
            p = base + 32 * k
            assert scol[p] == lcol[rowptr[r] + k]
            rows.append(l2g[r]); cols.append(l2g[scol[p]]); vv.append(vals[p])
    return sp.csr_matrix((vv, (rows, cols)), shape=(nv, nv))


@pytest.mark.parametrize("nranks", [1, 2, 3])
@pytest.mark.parametrize("reorder", [0, 1])
def test_rank_local_mesh(mesh, nranks, reorder):
    xy, cells = mesh
    nv = xy.shape[0]
    o = ShaktiOracle(xy, cells)
    rng = np.random.default_rng(0)
    Ke = rng.standard_normal((cells.shape[0], 9))
    ref = np.zeros(o.col.size)
    np.add.at(ref, o.slot.ravel(), Ke.ravel())
    Jref = sp.csr_matrix((ref, o.col, o.rowptr), shape=(nv, nv))
    owned_all, hms = [], []
    for r in range(nranks):
        hm = capi.HostMesh(xy, cells, r, nranks, reorder)
        hms.append(hm)
        l2g = hm.array("l2g")
        own = l2g[: hm.n_owned]
        owned_all.append(own)
        if reorder == 0 and nranks == 1:
            assert np.array_equal(l2g, np.arange(nv))
        lc, cl2g = hm.array("cells").reshape(-1, 3), hm.array("cell_l2g")
        assert np.array_equal(l2g[lc], cells[cl2g])                       # vertex order inside cells kept
        touched = np.isin(cells, own).any(axis=1)
        assert np.array_equal(np.sort(cl2g), np.nonzero(touched)[0])      # exactly the cells touching owned rows
        assert np.array_equal(hm.array("win_cell"), o.win_cell[own])      # winner by GLOBAL cell index
        win = hm.array("win").reshape(-1, 4)
        assert np.array_equal(l2g[win[np.arange(hm.n_owned), win[:, 3]]], own)
        # scatter through the slot table reproduces the oracle's CSR values on owned rows
        slot = hm.array("slot").reshape(9, -1)
        vals = np.zeros(hm.padded)
        m = slot >= 0
        np.add.at(vals, slot[m], Ke[cl2g].T[m])
        Jm = _sell_to_csr(hm, vals, nv)
        assert abs(Jm[own] - Jref[own]).max() < 1e-12
        scol, dp = hm.array("sell_col"), hm.array("diag_pos")
        assert np.array_equal(scol[dp], np.arange(hm.n_owned))
    allo = np.concatenate(owned_all)
    assert np.array_equal(np.sort(allo), np.arange(nv))                   # a partition of the dofs
    # halo maps are consistent pairwise: what r sends to s is what s expects from r, in order
    for r, hm in enumerate(hms):
        ranks, sptr, sidx = hm.array("nbr_rank"), hm.array("nbr_send_ptr"), hm.array("nbr_send_idx")
        l2g = hm.array("l2g")
        for k, s in enumerate(ranks):
            sent = l2g[sidx[sptr[k]: sptr[k + 1]]]
            h2 = hms[s]
            r2, recv, l2g2 = h2.array("nbr_rank"), h2.array("nbr_recv").reshape(-1, 2), h2.array("l2g")
            kk = int(np.nonzero(r2 == r)[0][0])
            assert np.array_equal(sent, l2g2[recv[kk, 0]: recv[kk, 0] + recv[kk, 1]])


def test_morton_order_is_local():
    """Rows of a 32-row slice should sit close together in space (SpMV gather locality)."""
    xy, cells = meshgen.rectangle(64, 64, 64.0, 64.0)
    hm = capi.HostMesh(xy, cells)
    l2g = hm.array("l2g")
    p = xy[l2g]
    spans = [np.ptp(p[s: s + 32], axis=0).max() for s in range(0, 32 * (len(p) // 32), 32)]
    assert np.median(spans) <= 8.0


def test_invalid_mesh_is_rejected():
    xy = np.zeros((3, 2))
    with pytest.raises(capi.ShaktiError):
        capi.HostMesh(xy, np.array([[0, 1, 5]], dtype=np.int32))


def test_product_never_imports_the_oracle():
    """oracle/ is test infrastructure: nothing under the product package may import it."""
    import ast
    pkg = ROOT / "shakti-fenics_b200"
    bad = []
    for f in list(pkg.rglob("*.py")):
        tree = ast.parse(f.read_text())
        for node in ast.walk(tree):
            names = []
            if isinstance(node, ast.Import):
                names = [a.name for a in node.names]
            elif isinstance(node, ast.ImportFrom) and node.module:
                names = [node.module]
            if any(n == "oracle" or n.startswith("oracle.") for n in names):
                bad.append(str(f))
    assert not bad, bad
    for f in (pkg / "csrc").glob("*"):
        if f.suffix in (".cu", ".cpp", ".h"):
            assert "oracle" not in f.read_text().lower(), f


# the rectangle, then the unstructured meshes of tests/unstructured.py (128-row blocks, 32-row blocks, refused)
PLAN_MESHES = [("rectangle", 1), ("rectangle", 2)] + [(n, k) for n in ("U0", "U32", "UA") for k in (1, 2)]


@pytest.mark.parametrize("name,nranks", PLAN_MESHES, ids=[str(k) if n == "rectangle" else f"{n}-{k}" for n, k in PLAN_MESHES])
def test_assembly_row_block_plan_emulated_in_numpy(mesh, name, nranks):
    """The plan behind assemble_blocks_kernel (csrc/prep.cpp build_assembly_blocks), executed in numpy exactly
    as the kernel does -- stage the block's cells, then gather per row through the incident-cell codes and the
    two-source codes -- must reproduce the plain scatter-add of the cell matrices, with no atomics.  On UA the
    plan of the rank that owns the 500-triangle fan is refused (the atomic fallback runs there instead)."""
    xy, cells = mesh if name == "rectangle" else unstructured.mesh(name)
    nv = xy.shape[0]
    o = ShaktiOracle(xy, cells)
    rng = np.random.default_rng(1)
    Ke = rng.standard_normal((cells.shape[0], 9))
    Fe = rng.standard_normal((cells.shape[0], 3))
    ref = np.zeros(o.col.size)
    np.add.at(ref, o.slot.ravel(), Ke.ravel())
    Jref = sp.csr_matrix((ref, o.col, o.rowptr), shape=(nv, nv))
    Fref = np.zeros(nv)
    np.add.at(Fref, cells.ravel(), Fe.ravel())
    refused = 0
    for r in range(nranks):
        hm = capi.HostMesh(xy, cells, r, nranks, 1)
        rb, nb, max_cells, max_verts, ok = hm.array("ab_info")
        if nranks == 1 and name != "rectangle":
            assert ((rb if ok else None), ok) == unstructured.PLAN[name, 1]
        if not ok:
            assert name == "UA"
            refused += 1
            continue
        assert rb in (32, 64, 128, 256) and max_cells <= 400
        l2g, lc, cl2g = hm.array("l2g"), hm.array("cells").reshape(-1, 3), hm.array("cell_l2g")
        eptr, elems, lv = hm.array("ab_eptr"), hm.array("ab_elems"), hm.array("ab_lv").reshape(-1, 3)
        hptr, halo = hm.array("ab_hptr"), hm.array("ab_halo")
        incptr, inc = hm.array("ab_incptr"), hm.array("ab_inc")
        src = hm.array("ab_src").view(np.uint32)
        sptr, rowptr = hm.array("slice_ptr"), hm.array("rowptr")
        vals = np.zeros(hm.padded)
        F = np.zeros(hm.n_owned)
        assert nb == (hm.n_owned + rb - 1) // rb and eptr[-1] == elems.size
        for B in range(nb):
            r0, r1 = B * rb, min(hm.n_owned, (B + 1) * rb)
            be = elems[eptr[B]:eptr[B + 1]]
            assert np.all(np.diff(be) > 0)
            # block-local vertex table = own rows then halo
            table = np.concatenate([np.arange(r0, r1), halo[hptr[B]:hptr[B + 1]]])
            assert table.size <= max_verts and np.array_equal(table[lv[eptr[B]:eptr[B + 1]]], lc[be])
            sK = np.concatenate([Fe[cl2g[be]], Ke[cl2g[be]]], axis=1)       # (cells in block, 12)
            for row in range(r0, r1):
                codes = inc[incptr[row]:incptr[row + 1]]
                le, a = codes >> 2, codes & 3
                F[row] = sK[le, a].sum()
                diag = sK[le, 3 + 4 * a].sum()
                base = sptr[row >> 5] + (row & 31)
                for k in range(rowptr[row + 1] - rowptr[row]):
                    pos = base + 32 * k
                    s2 = int(src[pos])
                    assert s2 != 0xFFFFFFFF
                    if s2 == 0xFFFEFFFE:
                        vals[pos] = diag
                    else:
                        ca, cb = s2 & 0xFFFF, s2 >> 16
                        vals[pos] = sK[ca >> 4, 3 + (ca & 15)] + (sK[cb >> 4, 3 + (cb & 15)] if cb != 0xFFFF else 0.0)
        own = l2g[: hm.n_owned]
        assert np.allclose(F, Fref[own], rtol=1e-13, atol=1e-13)
        assert abs(_sell_to_csr(hm, vals, nv)[own] - Jref[own]).max() < 1e-12
    assert refused == (1 if name == "UA" else 0)          # exactly the rank with the fan


def test_symmetric_heap_allocator_selftest():
    """The first-fit allocator that places halo staging slots and flags in the peer-mapped heap (csrc/comm.cu):
    alignment, no overlap of live blocks, double frees refused, full coalescing -- host logic, no GPU needed."""
    import ctypes as C
    lib = capi.load()
    for heap, rounds in ((1 << 20, 4000), (256 << 20, 20000), (4096, 200)):
        bad = C.c_int32(-1)
        assert lib.shakti_host_heap_selftest(C.c_int64(heap), C.c_int32(rounds), C.byref(bad)) == 0
        assert bad.value == 0, (heap, rounds, bad.value)


def _rows_match_oracle(xy, cells, nranks):
    nv = xy.shape[0]
    rp, col = csr_pattern(nv, cells)
    owned = []
    for r in range(nranks):
        hm = capi.HostMesh(xy, cells, r, nranks)
        l2g, no = hm.array("l2g"), hm.n_owned
        owned.append(l2g[:no])
        rowptr, lcol = hm.array("rowptr"), hm.array("col")
        for i in range(no):
            assert np.array_equal(np.sort(l2g[lcol[rowptr[i]:rowptr[i + 1]]]), col[rp[l2g[i]]:rp[l2g[i] + 1]])
        hm.array("ab_eptr")                      # the assembly plan builds (or reports the atomic fallback)
    assert np.array_equal(np.sort(np.concatenate(owned)), np.arange(nv))     # ownership is a partition


@pytest.mark.parametrize("kind", ["holes", "duplicated-cell", "tiny"])
def test_odd_meshes_preprocess_consistently(kind):
    """Ragged inputs: meshes with holes (dropped cells, unreferenced nodes pruned as DOLFINx does), a duplicated cell
    (three cells on an edge: the row-block plan must step aside, not miscount) and meshes with fewer rows than a
    SELL slice / than ranks -- every owned row's pattern equals the oracle's on 1, 2 and 3 ranks."""
    rng = np.random.default_rng(5)
    for trial in range(8):
        nx, ny = (int(rng.integers(1, 3)), int(rng.integers(1, 3))) if kind == "tiny" else (int(rng.integers(2, 9)), int(rng.integers(2, 9)))
        xy, cells = meshgen.rectangle(nx, ny, 1.0, 1.0, jitter=0.2, seed=trial, diagonal="random")
        xy, cells = meshgen.scramble(xy, cells, seed=trial)
        if kind == "holes":
            keep = rng.random(cells.shape[0]) > 0.4
            keep[0] = True
            cells = cells[keep]
            used = np.zeros(xy.shape[0], bool)
            used[cells.ravel()] = True
            cells = np.ascontiguousarray((np.cumsum(used) - 1)[cells], dtype=np.int32)
            xy = np.ascontiguousarray(xy[used])
        if kind == "duplicated-cell":
            cells = np.ascontiguousarray(np.vstack([cells, cells[:1]]))
        for nranks in (1, 2, 3):
            if nranks <= xy.shape[0]:
                _rows_match_oracle(xy, cells, nranks)


def test_unreferenced_vertex_is_refused():
    """A node no cell refers to would be an empty Jacobian row (singular system).  DOLFINx never creates such a dof;
    the library refuses the mesh with a message naming the vertex (and the .msh reader prunes such nodes)."""
    xy, cells = meshgen.rectangle(3, 3, 1.0, 1.0)
    xy2 = np.vstack([xy, [[9.0, 9.0]]])
    with pytest.raises(capi.ShaktiError) as e:
        capi.HostMesh(xy2, cells)
    assert "vertex 16 belongs to no cell" in str(e.value)
    for rank in (0, 1):                          # every rank of a job refuses it (no rank is left waiting)
        with pytest.raises(capi.ShaktiError):
            capi.HostMesh(xy2, cells, rank, 2)


def test_host_entry_points_validate_cell_ids():
    """Caller data reaches the host-only entry points unchecked by any shakti_create: a vertex id outside
    [0, n_vert) must come back as an error, not as a write outside the arrays."""
    xy, cells = meshgen.rectangle(3, 3, 1.0, 1.0)
    nv = xy.shape[0]
    for bad_id in (nv, -1, 2**31 - 1):
        bad = cells.copy()
        bad[4, 1] = bad_id
        with pytest.raises(capi.ShaktiError):
            capi.host_csr_pattern(nv, bad)
        with pytest.raises(capi.ShaktiError):
            capi.host_locate_dirichlet(nv, bad, np.ones(nv, bool))
        with pytest.raises(capi.ShaktiError):
            capi.HostMesh(xy, bad)


def test_degenerate_geometry_is_refused():
    """A cell of zero area (or a NaN coordinate) makes 1/det J infinite in every kernel; the mesh is refused with the
    cell named (the reference would carry NaNs into its first Newton solve)."""
    xy, cells = meshgen.rectangle(3, 3, 1.0, 1.0)
    flat = xy.copy()
    c = cells[5]
    flat[c[2]] = flat[c[0]]                                # two vertices of a cell coincide: zero area
    with pytest.raises(capi.ShaktiError) as e:
        capi.HostMesh(flat, cells)
    assert "zero area" in str(e.value)
    nan = xy.copy()
    nan[7, 0] = np.nan
    with pytest.raises(capi.ShaktiError):
        capi.HostMesh(nan, cells)
    capi.HostMesh(xy, cells)                               # the undisturbed mesh is fine
