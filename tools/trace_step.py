"""One C4 time step under torch.profiler (CUDA activity), once with each of two builds of the library, each in a run
of its own process.  Summarises the device time of the kernels around the AMG V-cycle's seams and the time the GPU
sits idle between the start of each Newton solve's fine-smoother refresh and the solve's first smoothing sweep (the
host round trip of a refresh that reads its bound back).  Writes the summary, and the chrome traces next to it.

  python tools/trace_step.py --base shakti-fenics_b200/lib/base/libshakti_b200.so [--new ...] \\
      [--out profiles/r3_cycle_seams_trace.json] [--trace-dir DIR]
"""
import argparse
import json
import subprocess
import sys
import tempfile
from collections import defaultdict
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
# kernels whose time the summary lists (substring of the demangled name)
WATCH = ("amg_dinv_kernel", "amg_gershgorin_kernel", "amg_fine_refresh_kernel", "amg_cheby_coef_kernel", "readback_kernel",
         "d2f_kernel", "f2d_kernel", "amg_cheby_first_kernel", "amg_cycle_entry_kernel", "restrict_cheby_first_kernel",
         "amg_cheby_kernel", "spmv_sell_kernel")
REFRESH = ("amg_gershgorin_kernel", "amg_fine_refresh_kernel")


def worker(lib, nside, warmup, trace):
    sys.path.insert(0, str(ROOT))
    sys.path.insert(0, str(ROOT / "shakti-fenics_b200"))
    import torch
    from shakti_b200 import capi, configs
    capi.LIB_PATH = Path(lib).resolve()
    case = configs.dofs16m(nside=nside, nsteps=warmup + 4)
    m = capi.Model(case.xy, case.cells, precond="amg", linear_rtol=1e-12)     # bench.py's defaults
    configs.apply_case(m, case)
    dts = case.dts()
    m.run(dts[:warmup])              # 3 (odd): the traced step keeps the hierarchy of the one before (amg_refresh_every = 2)
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        its, ms = m.run_timed(dts[warmup:warmup + 1])
        torch.cuda.synchronize()
    prof.export_chrome_trace(str(trace))
    m.close()
    ev = [e for e in json.loads(Path(trace).read_text())["traceEvents"] if e.get("cat") == "kernel"]
    ev.sort(key=lambda e: e["ts"])
    per = defaultdict(lambda: [0, 0.0])
    for e in ev:
        for w in WATCH:
            if w in e["name"]:
                key = w if w not in ("amg_cheby_kernel", "spmv_sell_kernel") else e["name"].split("(")[0]
                per[key][0] += 1
                per[key][1] += e["dur"]
    # idle GPU time from each fine-smoother refresh (the first refresh kernel of a solve on the fine level) to the first
    # Chebyshev sweep that follows it
    gaps = []
    i = 0
    while i < len(ev):
        if any(r in ev[i]["name"] for r in REFRESH):
            j = i
            while j < len(ev) and "amg_cheby_kernel" not in ev[j]["name"]:
                j += 1
            if j < len(ev):
                idle, end = 0.0, ev[i]["ts"] + ev[i]["dur"]
                for e in ev[i + 1:j + 1]:
                    idle += max(0.0, e["ts"] - end)
                    end = max(end, e["ts"] + e["dur"])
                gaps.append(dict(refresh_kernel=ev[i]["name"].split("(")[0], refresh_us=ev[i]["dur"], kernels=j - i,
                                 idle_us=round(idle, 1)))
            i = j + 1
        else:
            i += 1
    busy = sum(e["dur"] for e in ev)
    span = ev[-1]["ts"] + ev[-1]["dur"] - ev[0]["ts"] if ev else 0.0
    return dict(lib=str(lib), newton=int(its[0]), step_ms_events=ms, kernels=len(ev), kernel_busy_ms=busy / 1e3,
                span_ms=span / 1e3, refresh_to_first_sweep=gaps,
                kernels_us={k: dict(launches=v[0], total_us=round(v[1], 1), mean_us=round(v[1] / v[0], 1))
                            for k, v in sorted(per.items())})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--base", default=str(ROOT / "shakti-fenics_b200" / "lib" / "base" / "libshakti_b200.so"))
    ap.add_argument("--new", default=str(ROOT / "shakti-fenics_b200" / "lib" / "libshakti_b200.so"))
    ap.add_argument("--nside", type=int, default=4000)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--trace-dir", default=tempfile.gettempdir(), help="where the chrome traces go")
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r3_cycle_seams_trace.json"))
    ap.add_argument("--worker", help=argparse.SUPPRESS)
    ap.add_argument("--trace", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.worker:
        print(json.dumps(worker(args.worker, args.nside, args.warmup, args.trace)), flush=True)
        return
    res = {}
    for side in ("base", "new"):
        trace = Path(args.trace_dir) / f"cycle_seams_{side}.pt.trace.json"
        out = subprocess.run([sys.executable, __file__, "--worker", getattr(args, side), "--trace", str(trace),
                              "--nside", str(args.nside), "--warmup", str(args.warmup)], capture_output=True, text=True)
        if out.returncode != 0:
            raise SystemExit(f"{side}: {out.stderr[-3000:]}")
        res[side] = json.loads(out.stdout.strip().splitlines()[-1])
        print(json.dumps({side: {k: v for k, v in res[side].items() if k != "refresh_to_first_sweep"}}), flush=True)
    res["what"] = ("one C4 step (after 3 warm-up steps: every solve on a lagged hierarchy) under torch.profiler with each library in its own process; "
                   "kernel device times and GPU idle time from each fine-smoother refresh to the next smoothing sweep")
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
