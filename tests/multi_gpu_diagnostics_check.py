"""Multi-GPU check of the water-budget diagnostics (one process per GPU): run under torchrun, e.g.
  python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29521 \
      tests/multi_gpu_diagnostics_check.py
Every rank records one row per converged Newton solve; the rows (summed / reduced over ranks on the device) must
equal the one-shot records taken on the same states, and rank 0 checks those against the 1-rank CPU oracle loaded
with the gathered state: sums to 1e-12 relative, minima and maxima exactly."""
import os
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
for p in (str(ROOT), str(ROOT / "shakti-fenics_b200"), str(ROOT / "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

from budget_reference import oracle_diagnostics  # noqa: E402

FLUXES = ("input", "closure", "storage", "outflow", "imbalance")


def record_errors(got, ref, cm):
    """Errors of a record `got` against `ref` (dicts keyed by capi.DIAGNOSTICS).  Area, volume and mean N are
    relative to themselves; the terms of the balance (and the residual, in the same units) relative to the
    budget scale |input| + cm |melt| + |closure| + |storage| + |outflow| -- the imbalance of a converged solve
    is rounding and has no scale of its own.  Minima and maxima must be equal (0 error)."""
    scale = abs(ref["input"]) + cm * abs(ref["melt"]) + abs(ref["closure"]) + abs(ref["storage"]) + abs(ref["outflow"])
    e = {k: abs(got[k] - ref[k]) / abs(ref[k]) for k in ("area", "water_volume", "N_mean")}
    e.update({k: abs(got[k] - ref[k]) / scale for k in FLUXES})
    e["melt"] = cm * abs(got["melt"] - ref["melt"]) / scale
    e["residual"] = abs(got["residual"] - ref["residual"]) / max(scale, abs(ref["residual"]))
    e.update({k: float(got[k] != ref[k]) for k in ("N_min", "N_max", "b_max")})
    return e


def oracle_record(o, model_fields, dt):
    """The oracle's record at a state read back from the library (caller numbering, whole mesh)."""
    for k in ("N", "N_n", "b", "melt_n"):
        getattr(o, k)[:] = model_fields[k]
    o.q[:] = model_fields["q"]
    return oracle_diagnostics(o, dt)


def main():
    import torch
    import torch.distributed as dist
    from common import make_case, make_model, make_oracle
    from shakti_b200 import capi
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
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

    c = make_case(nx=48, ny=32, seed=9)
    m = make_model(*c, device=local, precond="amg", linear_max_it=5000)
    o = make_oracle(*c) if rank == 0 else None
    cm = 1 / 917 - 1 / 1000
    dts = [360.0, 3600.0, 3600.0, 3600.0]
    m.record_diagnostics(len(dts))
    worst, ok, shots = {}, True, []
    for dt in dts:
        it, _ = m.newton_solve(dt)
        shot = m.diagnostics(dt)
        shots.append([shot[k] for k in capi.DIAGNOSTICS])
        fields = {k: gsum(m.get_field(k)) for k in ("N", "N_n", "b", "melt_n")}
        fields["q"] = gsum(m.get_flux())
        if rank == 0:
            for k, v in record_errors(shot, oracle_record(o, fields, dt), cm).items():
                worst[k] = max(worst.get(k, 0.0), v)
        m.update_q_melt()
        m.update_b(dt)
        m.copy_N_to_N_n()
    rows = m.read_diagnostics()
    shots = np.array(shots)
    same = rows.shape == (len(dts), len(capi.DIAGNOSTICS)) and np.array_equal(rows[:, 3:], shots[:, 3:])
    if rank == 0:
        good = same and all(v <= (0.0 if k in ("N_min", "N_max", "b_max") else 1e-12) for k, v in worst.items())
        ok &= good
        print(f"[{world} GPUs, SHAKTI_P2P={os.environ.get('SHAKTI_P2P', '1')}] records == one-shot: {same}; errors vs "
              "oracle " + " ".join(f"{k}={v:.1e}" for k, v in worst.items()) + ("  OK" if good else "  MISMATCH"),
              flush=True)
    m.close()
    capi.comm_finalize()
    dist.destroy_process_group()
    if rank == 0:
        print("MULTI_GPU_DIAGNOSTICS " + ("PASSED" if ok else "FAILED"), flush=True)
        sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
