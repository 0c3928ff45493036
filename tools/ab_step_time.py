"""Step time of two builds of the library on the same steps, with their outputs compared bit for bit.  C4 (bench.py's
default mesh and inputs: configs.dofs16m, 16M dofs) on one GPU.  Each library runs in its own worker process, which
builds the model, runs the warm-up steps and takes a snapshot; the workers then take turns (A, B, A, B, ...), each leg
rolled back to the snapshot and timed with shakti_run_timed.  Asserts that N, b, qx, qy and melt_n after every leg
are bitwise equal and that the Newton and Krylov iteration counts are identical, and writes the result with the GPU's
name, power limit and clock read in the same run.  No torch import (start-up time).

  python tools/ab_step_time.py --base shakti-fenics_b200/lib/base/libshakti_b200.so \\
      [--new shakti-fenics_b200/lib/libshakti_b200.so] [--nside 4000] [--steps 10] [--out profiles/r3_cycle_seams_ab.json]
"""
import argparse
import json
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
FIELDS = ("N", "b", "qx", "qy", "melt_n")


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [s.strip() for s in out.split(",")]
        return dict(gpu=name, power_limit=power, sm_max_clock=clock)
    except Exception as e:     # the timings stand without it; say why it is missing
        return dict(gpu=None, power_limit=None, sm_max_clock=None, gpu_query_error=repr(e))


def worker(args):
    """Serves legs on stdin ("leg <dir>") for one library; one JSON line per leg on stdout."""
    sys.path.insert(0, str(ROOT))
    sys.path.insert(0, str(ROOT / "shakti-fenics_b200"))
    from shakti_b200 import capi, configs
    capi.LIB_PATH = Path(args.worker).resolve()
    t0 = time.perf_counter()
    case = configs.dofs16m(nside=args.nside, nsteps=args.warmup + args.steps + 4)
    m = capi.Model(case.xy, case.cells, precond="amg", linear_rtol=1e-12)     # bench.py's defaults
    configs.apply_case(m, case)
    dts = case.dts()
    m.run(dts[:args.warmup])
    m.snapshot()
    print(json.dumps(dict(ready=True, lib=str(capi.LIB_PATH), setup_s=round(time.perf_counter() - t0, 1))), flush=True)
    for line in sys.stdin:
        cmd = line.split()
        if not cmd or cmd[0] != "leg":
            break
        m.rollback()
        st0 = m.stats()
        its, ms = m.run_timed(dts[args.warmup:args.warmup + args.steps])
        st1 = m.stats()
        for f in FIELDS:
            np.save(Path(cmd[1]) / f"{f}.npy", m.get_field(f))
        print(json.dumps(dict(ms_per_step=ms / args.steps, newton=[int(i) for i in its],
                              krylov=int(st1["linear_its"] - st0["linear_its"]),
                              launches_per_step=(st1["kernel_launches"] - st0["kernel_launches"]) / args.steps)), flush=True)
    m.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--base", required=False, default=str(ROOT / "shakti-fenics_b200" / "lib" / "base" / "libshakti_b200.so"))
    ap.add_argument("--new", default=str(ROOT / "shakti-fenics_b200" / "lib" / "libshakti_b200.so"))
    ap.add_argument("--nside", type=int, default=4000)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--scratch", default=str(Path(tempfile.gettempdir()) / "ab_step_time"), help="directory for the fields of every leg")
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r3_cycle_seams_ab.json"))
    ap.add_argument("--worker", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.worker:
        return worker(args)
    libs = dict(base=args.base, new=args.new)
    for k, p in libs.items():
        if not Path(p).exists():
            raise SystemExit(f"{k} library {p} not found")
    common = ["--nside", str(args.nside), "--steps", str(args.steps), "--warmup", str(args.warmup)]
    procs = {}
    for k, p in libs.items():      # set up one after the other: the first leg of one must not overlap the other's set-up
        procs[k] = subprocess.Popen([sys.executable, __file__, "--worker", p] + common, stdin=subprocess.PIPE,
                                    stdout=subprocess.PIPE, text=True)
        ready = json.loads(procs[k].stdout.readline())
        print(json.dumps(dict(side=k, **ready)), flush=True)
    legs, ref = [], None
    scratch = Path(args.scratch)
    try:
        for rep in range(args.repeats):
            for k in libs:
                d = scratch / f"{k}_{rep}"
                d.mkdir(parents=True, exist_ok=True)
                procs[k].stdin.write(f"leg {d}\n")
                procs[k].stdin.flush()
                line = procs[k].stdout.readline()
                if not line:
                    raise SystemExit(f"{k} worker ended early")
                leg = dict(side=k, **json.loads(line))
                fields = {f: np.load(d / f"{f}.npy") for f in FIELDS}
                if ref is None:
                    ref = (fields, leg["newton"], leg["krylov"])
                leg["fields_equal"] = all(np.array_equal(fields[f], ref[0][f]) for f in FIELDS)
                leg["iterations_equal"] = leg["newton"] == ref[1] and leg["krylov"] == ref[2]
                legs.append(leg)
                print(json.dumps(leg), flush=True)
    finally:
        for p in procs.values():
            if p.poll() is None:
                p.stdin.close()
                p.wait(timeout=120)
    ms = {k: [x["ms_per_step"] for x in legs if x["side"] == k] for k in libs}
    med = {k: float(np.median(v)) for k, v in ms.items()}
    launches = {k: float(np.mean([x["launches_per_step"] for x in legs if x["side"] == k])) for k in libs}
    res = dict(
        what="C4 step time, parent library (base) against this one (new): same seeded steps rolled back before every "
             "leg, legs alternating, each library in its own process (shakti_run_timed)",
        **gpu_info(), nside=args.nside, steps_per_leg=args.steps,
        ms_per_step_base=ms["base"], ms_per_step_new=ms["new"], median_base=med["base"], median_new=med["new"],
        change_pct=float(100.0 * (med["new"] / med["base"] - 1.0)),
        launches_per_step_base=launches["base"], launches_per_step_new=launches["new"],
        newton_its=ref[1], krylov_its=ref[2],
        fields_bitwise_equal=all(x["fields_equal"] for x in legs),
        iterations_equal=all(x["iterations_equal"] for x in legs), legs=legs)
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(res, indent=1) + "\n")
    print(json.dumps({k: v for k, v in res.items() if k != "legs"}), flush=True)
    assert res["fields_bitwise_equal"], "fields differ between the libraries"
    assert res["iterations_equal"], "Newton / Krylov iteration counts differ between the libraries"


if __name__ == "__main__":
    main()
