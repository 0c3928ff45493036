"""Multi-GPU check of moulins (one process per GPU): run under torchrun, e.g.
  python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29531 \
      tests/multi_gpu_moulin_check.py
Moulins sit on partition-boundary vertices (the ghosts of each rank) and on interior vertices, two of them twice.
Before the communicator exists every rank runs the same case on one GPU; then the ranks together must give that
residual on every owned row (1e-14 of max |F|), the same Newton counts over 4 steps with fields equal to 1e-9, and
the same water-budget records up to the order of the reduction (1e-12 of the budget scale, extrema exactly)."""
import os
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
for p in (str(ROOT), str(ROOT / "shakti-fenics_b200"), str(ROOT / "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

from multi_gpu_diagnostics_check import record_errors  # noqa: E402

DT = 3600.0
DAY = 86400.0
T0 = 14 * 3600.0
DTS = [360.0, DT, DT, DT]


def moulins_on_the_cut(c, world):
    """Caller ids: up to 4 ghosts of every rank (vertices on the partition boundary, owned elsewhere), 4 interior
    vertices, and the first two again; diurnal hydrographs."""
    from shakti_b200 import capi, configs
    xy, cells, _, bc, _ = c
    rng = np.random.default_rng(5)
    picked = []
    for r in range(world):
        h = capi.HostMesh(xy, cells, rank=r, nranks=world)
        ghosts = np.setdiff1d(h.array("l2g")[h.n_owned:], bc)
        picked += rng.choice(ghosts, min(4, ghosts.size), replace=False).tolist()
    free = np.setdiff1d(np.arange(xy.shape[0]), np.concatenate([bc, picked]))
    v = picked + rng.choice(free, 4, replace=False).tolist()
    v += v[:2]
    q = rng.uniform(0.1, 0.5, len(v))
    return [int(a) for a in v], [configs.diurnal_hydrograph(qq, 1.2) for qq in q]


def run(m, vertex, tables):
    """residual at T0 + DT, then 4 steps with a budget record each -> (F, its, fields, rows)"""
    m.set_moulins(vertex, [t for t, _ in tables], [q for _, q in tables], period=DAY)
    m.set_time(T0)
    F = m.assemble(DT, want_J=False)[0]
    m.record_diagnostics(len(DTS))
    its = []
    for dt in DTS:
        it, _ = m.newton_solve(dt)
        m.update_q_melt()
        m.update_b(dt)
        m.copy_N_to_N_n()
        its.append(it)
    fields = {k: m.get_field(k) for k in ("N", "b", "qx", "qy")}
    return F, its, fields, m.read_diagnostics()


def main():
    import torch
    import torch.distributed as dist
    from common import make_case, make_model
    from shakti_b200 import capi
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    c = make_case(nx=48, ny=32, seed=9)
    vertex, tables = moulins_on_the_cut(c, world)
    opts = dict(device=local, precond="amg", linear_max_it=5000)
    one = make_model(*c, **opts)                       # before comm_init: a one-GPU model
    F1, its1, f1, rows1 = run(one, vertex, tables)
    one.close()

    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
    if rank == 0:
        uid = torch.tensor(list(capi.comm_unique_id()), dtype=torch.uint8, device="cuda")
    dist.broadcast(uid, 0)
    capi.comm_init(bytes(uid.cpu().tolist()), rank, world, local)

    def gsum(a):
        t = torch.from_numpy(np.ascontiguousarray(a)).cuda()
        dist.all_reduce(t)
        return t.cpu().numpy()

    m = make_model(*c, **opts)
    owned = m.owned()
    F, its, f, rows = run(m, vertex, tables)
    eF = float(np.max(np.abs(F[owned] - F1[owned])) / np.max(np.abs(F1)))
    fields = {k: gsum(v) for k, v in f.items()}
    eX = max(float(np.max(np.abs(fields[k] - f1[k])) / np.max(np.abs(f1[k]))) for k in fields)
    cm = 1 / 917 - 1 / 1000
    worst = {}
    for a, b in zip(rows, rows1):
        e = record_errors(dict(zip(capi.DIAGNOSTICS, a)), dict(zip(capi.DIAGNOSTICS, b)), cm)
        for k, v in e.items():
            worst[k] = max(worst.get(k, 0.0), v)
    ok_rank = (eF <= 1e-14 and its == its1 and eX <= 1e-9 and rows.shape == rows1.shape
               and all(v <= (0.0 if k in ("N_min", "N_max", "b_max") else 1e-12) for k, v in worst.items()))
    print(f"[rank {rank}/{world}, SHAKTI_P2P={os.environ.get('SHAKTI_P2P', '1')}] moulins on {len(set(vertex))} vertices; "
          f"F err {eF:.1e}; newton {its} vs 1 GPU {its1}; fields err {eX:.1e}; records "
          + " ".join(f"{k}={v:.1e}" for k, v in worst.items()) + ("  OK" if ok_rank else "  MISMATCH"), flush=True)
    ok = bool(gsum(np.array([0.0 if ok_rank else 1.0]))[0] == 0.0)
    m.close()
    capi.comm_finalize()
    dist.destroy_process_group()
    if rank == 0:
        print("MULTI_GPU_MOULINS " + ("PASSED" if ok else "FAILED"), flush=True)
        sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
