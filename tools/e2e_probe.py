"""Where does the end-to-end path lose time?  One model, the same K steps with and without the host copies, at a
set D2H chunk size."""
import os, sys, time, json
from pathlib import Path
ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT)); sys.path.insert(0, str(ROOT / "shakti-fenics_b200"))
import torch
from shakti_b200 import capi, configs

nside = int(sys.argv[1]) if len(sys.argv) > 1 else 4000
K = int(sys.argv[2]) if len(sys.argv) > 2 else 6
case = configs.dofs16m(nside=nside, nsteps=200)
m = capi.Model(case.xy, case.cells)
configs.apply_case(m, case)
dts = case.dts()
m.run(dts[:3])
own = m.owned()
n = own.size
h_in = capi.PinnedArray(n); h_in.array[:] = case.fields["inputs"][own]
sets = [[capi.PinnedArray(n) for _ in range(4)] for _ in range(2)]
step = 3

def run(label, chunk, use_in, use_out):
    global step
    os.environ["SHAKTI_D2H_CHUNK_MB"] = str(chunk)
    torch.cuda.synchronize()
    st0 = m.stats()
    first = step
    t0 = time.perf_counter()
    nits = []
    for i in range(K):
        outs = [b.array.ctypes.data for b in sets[i % 2]] if use_out else [None] * 4
        nits.append(m.step_host_async(dts[step], h_in.array.ctypes.data if use_in else None, *outs, owned_only=True)[0])
        step += 1
    m.wait_outputs()
    torch.cuda.synchronize()
    ms = 1e3 * (time.perf_counter() - t0) / K
    st1 = m.stats()
    print(json.dumps(dict(label=label, chunk_mb=chunk, h2d=use_in, d2h=use_out, ms_per_step=round(ms, 2),
                          first_step=first, newton=nits, krylov_per_step=(st1["linear_its"] - st0["linear_its"]) / K,
                          refreshes=st1["amg_refreshes"] - st0["amg_refreshes"])), flush=True)

for rep in range(3):
    run("no copies", 8, False, False)
    run("both", 8, True, True)
