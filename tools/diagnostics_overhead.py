"""What does recording the water budget cost?  C4 (bench.py's default mesh and inputs: configs.dofs16m, 16M dofs) on
one GPU: the same seeded steps (state rolled back before every leg) with shakti_record_diagnostics off and on,
alternating 3x each, each leg timed with shakti_run_timed.  Checks that the fields after every leg are bitwise the
same with recording on and off and that every record closes the budget, and writes the result with the GPU's name and
power limit read in the same run.  No torch import (start-up time).

  python tools/diagnostics_overhead.py [--nside 4000] [--steps 10] [--out profiles/r3_diagnostics_overhead.json]
"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "shakti-fenics_b200"))
from shakti_b200 import capi, configs  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [s.strip() for s in out.split(",")]
        return dict(gpu=name, power_limit=power, sm_max_clock=clock)
    except Exception as e:     # the timings stand without it; say why it is missing
        return dict(gpu=None, power_limit=None, sm_max_clock=None, gpu_query_error=repr(e))


def budget_error(rows):
    """max over records of |outflow - (input - cm melt + closure + storage + imbalance)| / budget scale"""
    d = {k: rows[:, i] for i, k in enumerate(capi.DIAGNOSTICS)}
    cm = 1 / 917 - 1 / 1000
    scale = np.abs(d["input"]) + cm * np.abs(d["melt"]) + np.abs(d["closure"]) + np.abs(d["storage"]) + np.abs(d["outflow"])
    rhs = d["input"] - cm * d["melt"] + d["closure"] + d["storage"] + d["imbalance"]
    return float(np.max(np.abs(d["outflow"] - rhs) / scale))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nside", type=int, default=4000)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r3_diagnostics_overhead.json"))
    args = ap.parse_args()
    t0 = time.perf_counter()
    case = configs.dofs16m(nside=args.nside, nsteps=args.warmup + args.steps + 4)
    m = capi.Model(case.xy, case.cells, precond="amg", linear_rtol=1e-12)     # bench.py's defaults
    configs.apply_case(m, case)
    dts = case.dts()
    m.run(dts[:args.warmup])
    m.snapshot()
    setup_s = time.perf_counter() - t0
    legs, ref, rows_all = [], None, []
    for rep in range(args.repeats):
        for on in (False, True):
            m.rollback()
            m.record_diagnostics(args.steps if on else 0)
            l0 = m.stats()["kernel_launches"]
            its, ms = m.run_timed(dts[args.warmup:args.warmup + args.steps])
            launches = m.stats()["kernel_launches"] - l0
            rows = m.read_diagnostics() if on else None
            fields = (m.get_field("N"), m.get_field("b"))
            if ref is None:
                ref = fields
            same = all(np.array_equal(a, b) for a, b in zip(fields, ref))
            legs.append(dict(recording=on, ms_per_step=ms / args.steps, newton=int(sum(its)),
                             launches_per_step=launches / args.steps, fields_equal_first_leg=same))
            if on:
                rows_all.append(rows)
            print(json.dumps(legs[-1]), flush=True)
    m.record_diagnostics(0)
    off = [x["ms_per_step"] for x in legs if not x["recording"]]
    on = [x["ms_per_step"] for x in legs if x["recording"]]
    rows = np.concatenate(rows_all)
    res = dict(
        what="C4 step time with water-budget recording off and on (shakti_run_timed, same steps, alternating legs)",
        **gpu_info(), n_vert=int(case.n_vert), n_cell=int(case.cells.shape[0]), steps_per_leg=args.steps,
        ms_per_step_off=off, ms_per_step_on=on,
        median_off=float(np.median(off)), median_on=float(np.median(on)),
        overhead_pct=float(100.0 * (np.median(on) / np.median(off) - 1.0)),
        extra_launches_per_step=float(np.mean([x["launches_per_step"] for x in legs if x["recording"]])
                                      - np.mean([x["launches_per_step"] for x in legs if not x["recording"]])),
        fields_equal=all(x["fields_equal_first_leg"] for x in legs),
        records_bitwise_repeatable=all(np.array_equal(r, rows_all[0]) for r in rows_all),
        max_budget_error=budget_error(rows), setup_s=round(setup_s, 1), legs=legs)
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(res, indent=1) + "\n")
    print(json.dumps({k: v for k, v in res.items() if k != "legs"}), flush=True)
    m.close()


if __name__ == "__main__":
    main()
