"""Device time and fraction of the HBM peak of the one-thread-per-row SELL kernels of the V-cycle: smoother, residual,
restriction and prolongation of every AMG level of >= 300 000 rows.  C4 (bench.py's default mesh and inputs:
configs.dofs16m, 16M dofs) on one GPU, after the warm-up steps; each kernel is launched as the cycle launches it,
`--reps` times back to back between CUDA events (shakti_time_amg_level_kernel), the matrices are far larger than L2.
Writes the result with the GPU's name, power limit and clock read in the same run.  No torch import.

A kernel is listed when its matrix has >= 300 000 rows (smaller ones run the block-per-slice kernels).  Algorithmic
bytes per launch (vb = bytes per value of the kernel's matrix, xb = bytes per vector entry; nnz, rows, cols of the
kernel's matrix):
  smoother      (vb+4) nnz + 7 xb rows   reads dinv, b, x (twice: gather and update), d; writes d, x_out
  residual      (vb+4) nnz + 3 xb rows   reads b, x; writes r
  restriction   (vb+4) nnz + xb cols + xb rows     reads r; writes b_c
                + 2 xb rows when fused with the coarse level's first Chebyshev step (reads dinv_c, writes x_c)
  prolongation  (vb+4) nnz + xb cols + 2 xb rows   reads x_c; reads and writes x

  python tools/sell_kernels.py [--lib shakti-fenics_b200/lib/libshakti_b200.so] [--nside 4000] [--out FILE]
"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "shakti-fenics_b200"))
from shakti_b200 import capi, configs  # noqa: E402

WIDE_ROWS = 300000        # levels with fewer rows run the block-per-slice kernels
VECTORS = {"smoother": (7, 0), "residual": (3, 0), "restriction": (1, 1), "prolongation": (2, 1)}   # per row, per column


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [s.strip() for s in out.split(",")]
        return dict(gpu=name, power_limit=power, sm_max_clock=clock)
    except Exception as e:     # the timings stand without it; say why it is missing
        return dict(gpu=None, power_limit=None, sm_max_clock=None, gpu_query_error=repr(e))


def hbm_peak():
    f = ROOT / "MEASURED_PEAKS.json"
    if f.exists():
        return float(json.loads(f.read_text())["hbm_gbs"]), "measured copy bandwidth (MEASURED_PEAKS.json)"
    return 6547.5, "measured copy bandwidth of the B200 of profiles/r1_bench_n8.json"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", default=str(ROOT / "shakti-fenics_b200" / "lib" / "libshakti_b200.so"))
    ap.add_argument("--nside", type=int, default=4000)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--out", help="JSON file for the result (default: print only)")
    args = ap.parse_args()
    capi.LIB_PATH = Path(args.lib).resolve()
    peak, peak_src = hbm_peak()
    t0 = time.perf_counter()
    case = configs.dofs16m(nside=args.nside, nsteps=args.warmup + 4)
    m = capi.Model(case.xy, case.cells, precond="amg", linear_rtol=1e-12)     # bench.py's defaults
    configs.apply_case(m, case)
    m.run(case.dts()[:args.warmup])
    setup_s = time.perf_counter() - t0
    rows_out = []
    for lvl in range(m.stats()["amg_levels"]):
        for k in capi.Model.AMG_LEVEL_KERNELS:
            try:
                r = m.time_amg_level_kernel(lvl, k, reps=1)
            except capi.ShaktiError:
                continue
            if r["rows"] < WIDE_ROWS:
                continue
            r = m.time_amg_level_kernel(lvl, k, reps=args.reps)
            per_row, per_col = VECTORS[k]
            if k == "restriction" and r["fused"]:
                per_row += 2
            xb = r["vector_bytes"]
            by = (r["value_bytes"] + 4) * r["nnz"] + xb * (per_row * r["rows"] + per_col * r["cols"])
            gbs = by / 1e9 / (r["ms"] / 1e3)
            rows_out.append(dict(level=lvl, kernel=k, us=1e3 * r["ms"], rows=r["rows"], cols=r["cols"], nnz=r["nnz"],
                                 max_width=r["max_width"], value_bytes=r["value_bytes"], vector_bytes=xb,
                                 fused=r["fused"], algorithmic_GB=by / 1e9, GBps=gbs, frac=gbs / peak))
            print(json.dumps(rows_out[-1]), flush=True)
    m.close()
    res = dict(what="one-thread-per-row SELL kernels of the V-cycle at C4, mean device time of back-to-back launches "
                    "(CUDA events), algorithmic bytes over time against the HBM peak",
               lib=str(capi.LIB_PATH), **gpu_info(), nside=args.nside, reps=args.reps, setup_s=round(setup_s, 1),
               peak_GBps=peak, peak_source=peak_src, kernels=rows_out)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(res, indent=1) + "\n")
    print(json.dumps({k: v for k, v in res.items() if k != "kernels"}), flush=True)


if __name__ == "__main__":
    main()
