"""World-size-2 (and 3) emulation of the multi-GPU path on the CPU with the gloo backend: the
partition, owner-computes cell overlap and halo maps produced by the C library's host code
drive a numpy restatement of what each GPU rank does (halo exchange -> local SpMV, all-reduced
dots, nodal update ownership), and the result must equal the single-rank/global computation."""
import os
import sys
import socket
from pathlib import Path

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = Path(__file__).resolve().parent.parent
for p in (str(ROOT), str(ROOT / "shakti-fenics_b200"), str(ROOT / "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _halo_exchange(hm, v, rank):
    """owner -> ghost copies with point-to-point messages, as csrc/comm.cu does with NCCL."""
    ranks, sptr, sidx = hm.array("nbr_rank"), hm.array("nbr_send_ptr"), hm.array("nbr_send_idx")
    recv = hm.array("nbr_recv").reshape(-1, 2)
    reqs, bufs = [], []
    for k, peer in enumerate(ranks):
        out = torch.from_numpy(np.ascontiguousarray(v[sidx[sptr[k]: sptr[k + 1]]]))
        inn = torch.empty(int(recv[k, 1]), dtype=torch.float64)
        bufs.append((k, inn))
        reqs.append(dist.isend(out, int(peer)))
        reqs.append(dist.irecv(inn, int(peer)))
    for r in reqs:
        r.wait()
    for k, inn in bufs:
        v[recv[k, 0]: recv[k, 0] + recv[k, 1]] = inn.numpy()


def _worker(rank, world, port, q, mesh="rectangle"):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from common import case_on, make_case, make_oracle
        from shakti_b200 import capi
        import scipy.sparse as sp
        if mesh == "rectangle":
            c = make_case(nx=20, ny=14, seed=3)
        else:                                                # ragged partitions of an unstructured mesh
            import unstructured
            c = case_on(*unstructured.mesh(mesh), seed=3)
        o = make_oracle(*c)
        xy, cells = c[0], c[1]
        nv = xy.shape[0]
        F, vals = o.assemble(3600.0)
        J = o.jacobian_matrix(vals)
        hm = capi.HostMesh(xy, cells, rank, world, 1)
        l2g = hm.array("l2g")
        no, nl = hm.n_owned, hm.n_local
        # local operator: owned rows x local columns, from the global matrix
        g2l = -np.ones(nv, dtype=np.int64)
        g2l[l2g] = np.arange(nl)
        Jl = J[l2g[:no]].tocoo()
        assert (g2l[Jl.col] >= 0).all()                      # every column of an owned row is local (owned or ghost)
        Aloc = sp.csr_matrix((Jl.data, (Jl.row, g2l[Jl.col])), shape=(no, nl))
        # owner-computes: local cells assemble the owned rows completely
        lc, cl2g = hm.array("cells").reshape(-1, 3), hm.array("cell_l2g")
        Fe, _ = o.element_FJ(3600.0)
        Floc = np.zeros(nl)
        np.add.at(Floc, lc.ravel(), Fe[cl2g].ravel())
        Fglob = np.zeros(nv)
        np.add.at(Fglob, cells.ravel(), Fe.ravel())          # all cells, no Dirichlet handling
        own = l2g[:no]
        assert np.allclose(Floc[:no], Fglob[own], rtol=1e-12, atol=1e-12 * np.abs(Fglob).max())
        # distributed y = J x with halo exchange
        rng = np.random.default_rng(0)
        xg = rng.standard_normal(nv)
        xl = np.zeros(nl)
        xl[:no] = xg[own]
        _halo_exchange(hm, xl, rank)
        assert np.array_equal(xl, xg[l2g])                   # ghosts received the owners' values
        y = Aloc @ xl
        assert np.allclose(y, (J @ xg)[own], rtol=1e-13, atol=1e-13 * np.abs(J @ xg).max())
        # distributed Jacobi-preconditioned BiCGStab with all-reduced dots
        def dot(a, b):
            t = torch.tensor([float(a @ b)], dtype=torch.float64)
            dist.all_reduce(t)
            return float(t.item())

        def matvec(v):
            w = np.zeros(nl)
            w[:no] = v
            _halo_exchange(hm, w, rank)
            return Aloc @ w

        dinv = 1.0 / J.diagonal()[own]
        b = F[own]
        # norms over the rows that are not Dirichlet rows: those hold N - N_bdry, orders of magnitude above the
        # interior residual, and would let the interior stop early and hide its error
        inner = np.ones(nv, dtype=bool)
        inner[c[3]] = False
        mine = inner[own]
        x = np.zeros(no)
        r = b.copy(); r0 = r.copy(); p = np.zeros(no); v = np.zeros(no)
        rho = alpha = om = 1.0
        bn = np.sqrt(dot(b[mine], b[mine]))
        for it in range(2000):
            rho_n = dot(r0, r)
            beta = (rho_n / rho) * (alpha / om)
            p = r + beta * (p - om * v)
            ph = dinv * p
            v = matvec(ph)
            alpha = rho_n / dot(r0, v)
            s = r - alpha * v
            sh = dinv * s
            t = matvec(sh)
            om = dot(t, s) / dot(t, t)
            x += alpha * ph + om * sh
            r = s - om * t
            rho = rho_n
            if np.sqrt(dot(r, r)) <= 1e-12 * bn:
                break
        import scipy.sparse.linalg as spla
        ref = spla.splu(J.tocsc()).solve(F)
        # true residual of the distributed solution: interior rows to the stopping tolerance (their rounding in
        # the Dirichlet rows, x = N - N_bdry of up to 2e4, is far above it and is checked row by row)
        rt = b - matvec(x)
        assert np.sqrt(dot(rt[mine], rt[mine])) <= 1e-11 * bn
        assert np.all(np.abs(rt[~mine]) <= 1e-14 * np.abs(b[~mine]).max(initial=0.0))
        # against LU on the interior rows: 8e-13 on the rectangle, 4e-12 on U32 (in a one-rank restatement)
        err = np.abs(x - ref[own])[mine].max() / np.abs(ref[inner]).max()
        assert err < 1e-10, err
        # nodal-update ownership: every vertex is owned exactly once and its winning cell is local
        wc = hm.array("win_cell")
        assert np.array_equal(wc, o.win_cell[own]) and np.isin(wc, cl2g).all()
        cnt = torch.zeros(nv, dtype=torch.float64)
        cnt[torch.from_numpy(own.astype(np.int64))] += 1
        dist.all_reduce(cnt)
        assert bool((cnt == 1).all())
        q.put((rank, "ok"))
    except Exception as e:  # noqa: BLE001
        import traceback
        q.put((rank, "FAIL " + "".join(traceback.format_exception(e))))
    finally:
        dist.destroy_process_group()


# the rectangle, then U32 of tests/unstructured.py (a fan of 320 triangles, graded Delaunay cells)
PARTITIONED = [(2, "rectangle"), (3, "rectangle"), (2, "U32"), (3, "U32")]


@pytest.mark.parametrize("world,mesh", PARTITIONED, ids=[str(w) if m == "rectangle" else f"{m}-{w}" for w, m in PARTITIONED])
def test_partitioned_path_equals_global(world, mesh):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q, mesh)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=300) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
    assert all(msg == "ok" for _, msg in res), res


def test_multi_gpu_check_script_imports_without_gpus():
    """tests/multi_gpu_check.py is launched by torchrun on >= 2 GPUs only; on any box it must at least import
    (paths, helper modules) so a one-GPU CI run still catches a broken script."""
    import importlib
    mod = importlib.import_module("multi_gpu_check")
    assert callable(mod.main)
