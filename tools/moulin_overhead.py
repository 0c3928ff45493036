"""What do moulins cost?  C4 (bench.py's mesh and inputs: configs.dofs16m, 16M dofs) on one GPU: the same seeded
steps (state and clock rolled back before every leg) with no moulins and with 1000 moulins carrying 48-knot periodic
hydrographs, alternating 3x each, each leg timed with shakti_run_timed.  The timed tables are zero, so both legs
solve the same problem bit for bit and the difference is the moulin kernel; one more leg with nonzero tables shows
what the forcing itself does to the Newton and Krylov work.  Also counts the kernel launches per step at C1 size
(configs.cooke2_like) with and without moulins, where one extra launch per assembly is a visible share of a
launch-bound step.  Writes the result with the GPU's name and power limit read in the same run.  No torch import.

  python tools/moulin_overhead.py [--nside 4000] [--steps 10] [--out profiles/r3_moulin_overhead.json]
"""
import argparse
import json
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "shakti-fenics_b200"))
sys.path.insert(0, str(ROOT / "tools"))
from diagnostics_overhead import gpu_info  # noqa: E402
from shakti_b200 import capi, configs  # noqa: E402


def random_moulins(case, bc, n, knots, seed, scale=1.0):
    """n moulins on seeded non-Dirichlet vertices, diurnal hydrographs of `knots` intervals, mean 0.05-0.5 m^3/s
    times `scale`.  scale = 0: every table is zero, so F, the Newton iteration and the fields are bitwise those
    without moulins and a timing difference is the cost of the moulin kernel alone (it does the same lookups)."""
    rng = np.random.default_rng(seed)
    v = rng.choice(np.setdiff1d(np.arange(case.n_vert), bc), n, replace=False)
    tables = [configs.diurnal_hydrograph(q, 1.2, knots_per_day=knots) for q in scale * rng.uniform(0.05, 0.5, n)]
    return v, [t for t, _ in tables], [q for _, q in tables]


def launches_per_step(m, dts):
    l0 = m.stats()["kernel_launches"]
    m.run(dts)
    return (m.stats()["kernel_launches"] - l0) / len(dts)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nside", type=int, default=4000)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--moulins", type=int, default=1000)
    ap.add_argument("--knots", type=int, default=48)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r3_moulin_overhead.json"))
    args = ap.parse_args()
    info = gpu_info()

    # C1 size: kernel launches per step (the same steps, with and without moulins)
    c1 = configs.cooke2_like(nsteps=12)
    c1.timesteps = np.linspace(0, 11 * 3600.0, 12)
    counts = {}
    for with_moulins in (False, True):
        m = configs.apply_case(capi.Model(c1.xy, c1.cells), c1)
        bc = m.locate_dirichlet(c1.meta["outflow_marker"])
        if with_moulins:
            m.set_moulins(*random_moulins(c1, bc, 60, 24, seed=3, scale=0.0), period=configs.DAY)
        dts = c1.dts()
        m.run(dts[:4])
        counts[with_moulins] = launches_per_step(m, dts[4:10])
        m.close()

    t0 = time.perf_counter()
    case = configs.dofs16m(nside=args.nside, nsteps=args.warmup + args.steps + 4)
    m = capi.Model(case.xy, case.cells, precond="amg", linear_rtol=1e-12)     # bench.py's defaults
    configs.apply_case(m, case)
    mo = random_moulins(case, case.bc_dofs, args.moulins, args.knots, seed=11, scale=0.0)
    mo_forcing = random_moulins(case, case.bc_dofs, args.moulins, args.knots, seed=11)
    dts = case.dts()
    m.set_time(12 * 3600.0)
    m.run(dts[:args.warmup])
    m.snapshot()
    setup_s = time.perf_counter() - t0
    legs, ref = [], {}
    for rep in range(args.repeats):
        for on in (False, True):
            m.rollback()
            if on:
                m.set_moulins(*mo, period=configs.DAY)
            else:
                m.set_moulins([], [], [])
            l0 = m.stats()["kernel_launches"]
            its, ms = m.run_timed(dts[args.warmup:args.warmup + args.steps])
            launches = m.stats()["kernel_launches"] - l0
            fields = (m.get_field("N"), m.get_field("b"))
            ref.setdefault(0, fields)
            same = all(np.array_equal(a, b) for a, b in zip(fields, ref[0]))
            legs.append(dict(moulins=args.moulins if on else 0, ms_per_step=ms / args.steps, newton=int(sum(its)),
                             launches_per_step=launches / args.steps, fields_equal_first_leg=same))
            print(json.dumps(legs[-1]), flush=True)
    # the same moulins with their nonzero tables: a different (harder) problem, reported for information
    m.rollback()
    m.set_moulins(*mo_forcing, period=configs.DAY)
    l0 = m.stats()["kernel_launches"]
    its, ms = m.run_timed(dts[args.warmup:args.warmup + args.steps])
    forced = dict(ms_per_step=ms / args.steps, newton=int(sum(its)),
                  launches_per_step=(m.stats()["kernel_launches"] - l0) / args.steps)
    off = [x["ms_per_step"] for x in legs if not x["moulins"]]
    on = [x["ms_per_step"] for x in legs if x["moulins"]]
    res = dict(
        what=f"C4 step time without and with {args.moulins} moulins ({args.knots}-knot periodic hydrographs, all zero, "
             "so the fields are bitwise those without moulins), shakti_run_timed, same steps rolled back, alternating "
             "legs; launches per step at C1 size with 60 zero-table moulins; and one leg with the tables nonzero",
        **info, n_vert=int(case.n_vert), n_cell=int(case.cells.shape[0]), steps_per_leg=args.steps,
        ms_per_step_without=off, ms_per_step_with=on,
        median_without=float(np.median(off)), median_with=float(np.median(on)),
        overhead_pct=float(100.0 * (np.median(on) / np.median(off) - 1.0)),
        extra_launches_per_step_c4=float(np.mean([x["launches_per_step"] for x in legs if x["moulins"]])
                                         - np.mean([x["launches_per_step"] for x in legs if not x["moulins"]])),
        newton_per_leg_without=[x["newton"] for x in legs if not x["moulins"]],
        newton_per_leg_with=[x["newton"] for x in legs if x["moulins"]],
        fields_equal=all(x["fields_equal_first_leg"] for x in legs),
        c1_n_vert=int(c1.n_vert), c1_launches_per_step_without=counts[False], c1_launches_per_step_with_60=counts[True],
        nonzero_tables_leg=forced,
        setup_s=round(setup_s, 1), legs=legs)
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(res, indent=1) + "\n")
    print(json.dumps({k: v for k, v in res.items() if k != "legs"}), flush=True)
    m.close()


if __name__ == "__main__":
    main()
