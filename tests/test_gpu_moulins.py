"""Moulins on the GPU: the residual term against the assembly without moulins, the hydrograph lookup, transient runs
against the CPU reference (tests/moulin_reference.py), rollback, the water budget, the no-moulin path, argument
validation, solvers.solve(md) on the SHMIP-like setup and the 2-GPU check."""
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
for p in (ROOT / "shakti-fenics_b200" / "source", ROOT / "shakti-fenics_b200" / "setups"):
    if str(p) not in sys.path:
        sys.path.insert(0, str(p))

from common import make_case, make_model, relinf  # noqa: E402
from moulin_reference import MoulinOracle, hydrograph, moulin_diagnostics  # noqa: E402
from multi_gpu_diagnostics_check import record_errors  # noqa: E402
from oracle.shakti_oracle import ShaktiOracle  # noqa: E402
from shakti_b200 import capi, configs  # noqa: E402

pytestmark = pytest.mark.gpu

DT = 3600.0
DAY = 86400.0
CM = 1 / 917 - 1 / 1000
T0 = 14 * 3600.0


def moulin_set(nv, bc, seed=1, n=10):
    """n moulins on distinct free vertices plus two more on the first two of them (duplicates), diurnal tables."""
    rng = np.random.default_rng(seed)
    v = rng.choice(np.setdiff1d(np.arange(nv), bc), n, replace=False)
    v = np.concatenate([v, v[:2]])
    return [(int(a), *configs.diurnal_hydrograph(q, 1.2)) for a, q in zip(v, rng.uniform(0.1, 0.5, v.size))]


def set_moulins(m, mo, period=DAY):
    m.set_moulins([v for v, _, _ in mo], [t for _, t, _ in mo], [q for _, _, q in mo], period=period)


def moulin_oracle(c, mo, t0):
    xy, cells, f, bc, N_bdry = c
    o = MoulinOracle(xy, cells)
    for k in ("z_b", "z_s", "G", "inputs", "storage", "b", "N_n", "melt_n"):
        getattr(o, k)[:] = f[k]
    o.q[:] = f["q"]
    o.set_dirichlet(bc, N_bdry)
    o.start()
    o.set_moulins(mo, DAY)
    o.t = t0
    return o


def state(m):
    return [m.get_field(k) for k in ("N", "b", "melt_n", "qx", "qy", "N_n")]


@pytest.mark.parametrize("kernel", [0, 1], ids=["row-block-gather", "cell-atomics"])
def test_assemble_difference_is_minus_q_on_moulin_rows(kernel):
    c = make_case(seed=3)
    mo = moulin_set(c[0].shape[0], c[3])
    a, b = make_model(*c, assembly_kernel=kernel), make_model(*c, assembly_kernel=kernel)
    try:
        set_moulins(a, mo)
        for m in (a, b):
            m.set_time(T0)
        Fa, Ja = a.assemble(DT)
        Fb, Jb = b.assemble(DT)
        q = a.moulin_discharge(T0 + DT)
        s = {}
        for (v, _, _), qk in zip(mo, q):          # per row, in the order given, from 0
            s[v] = s.get(v, 0.0) + qk
        rows = np.array(sorted(s))
        want = np.array([s[v] for v in rows])
        assert rows.size == len(mo) - 2 and want.min() > 0
        other = np.setdiff1d(np.arange(Fa.size), rows)
        scale = np.abs(Fb).max()
        if kernel == 0:
            # the row-block kernel sums in a fixed order: everything but the moulin term is bitwise the same
            ulp = np.spacing(np.maximum(np.abs(Fa[rows]), np.abs(Fb[rows])))
            assert np.all(np.abs((Fa[rows] - Fb[rows]) + want) <= ulp)
            assert np.array_equal(Fa[other], Fb[other])
            assert np.array_equal(Ja, Jb)
        else:
            # the cell kernel adds with floating-point atomics: its sums vary in the last bits from run to run
            assert np.all(np.abs((Fa[rows] - Fb[rows]) + want) <= 1e-13 * scale)
            assert np.all(np.abs(Fa[other] - Fb[other]) <= 1e-13 * scale)
            assert np.allclose(Ja, Jb, rtol=1e-13, atol=1e-13 * np.abs(Jb).max())
        # removing the moulins gives the assembly without them back
        a.set_moulins([], [], [])
        F0 = a.assemble(DT)[0]
        assert np.array_equal(F0, Fb) if kernel == 0 else np.all(np.abs(F0 - Fb) <= 1e-13 * scale)
    finally:
        a.close()
        b.close()


def test_moulin_discharge_matches_numpy():
    c = make_case(seed=1)
    rng = np.random.default_rng(4)
    mo = moulin_set(c[0].shape[0], c[3], seed=2)
    tk = np.sort(rng.uniform(-5e3, 7e4, 9))                     # irregular table, shorter than the period
    mo.append((mo[0][0], tk, rng.uniform(0.0, 4.0, tk.size)))
    m = make_model(*c)
    try:
        for period in (0.0, DAY):
            set_moulins(m, mo, period)
            ts = np.concatenate([np.linspace(-3 * DAY, 4 * DAY, 997), tk, tk + period, [tk[0] - period, -1e9, 1e9]])
            for t in ts:
                got = m.moulin_discharge(t)
                ref = np.array([hydrograph(tt, qq, t, period) for _, tt, qq in mo])
                assert np.all(np.abs(got - ref) <= 1e-15 * np.maximum(np.abs(ref), 1.0)), (period, t)
    finally:
        m.close()


def _transient(c, mo, dts, split):
    m = make_model(*c)
    set_moulins(m, mo)
    m.set_time(T0)
    if split:
        its = []
        for dt in dts:
            it, _ = m.newton_solve(dt)
            m.update_q_melt()
            m.update_b(dt)
            m.copy_N_to_N_n()
            its.append(it)
    else:
        its = list(m.run(dts))
    return m, its


def test_transient_diurnal_against_reference_run_and_split_path():
    c = make_case(seed=5)
    mo = moulin_set(c[0].shape[0], c[3])
    dts = ShaktiOracle.dt_schedule(np.linspace(0, 9 * DT, 10))
    o = moulin_oracle(c, mo, T0)
    its_o = [o.step(dt)[0] for dt in dts]
    a, its_a = _transient(c, mo, dts, split=False)
    b, its_b = _transient(c, mo, dts, split=True)
    try:
        assert its_a == its_o and its_b == its_o, (its_a, its_b, its_o)
        assert a.get_time() == o.t == b.get_time()
        assert relinf(a.get_field("N"), o.N) <= 1e-8 and relinf(a.get_field("b"), o.b) <= 1e-8
        assert relinf(a.get_flux(), o.q) <= 1e-7
        for x, y in zip(state(a), state(b)):
            assert np.array_equal(x, y)
    finally:
        a.close()
        b.close()


def test_snapshot_rollback_restores_fields_and_time():
    c = make_case(seed=6)
    mo = moulin_set(c[0].shape[0], c[3])
    m = make_model(*c)
    try:
        set_moulins(m, mo)
        m.set_time(T0)
        m.run([360.0, DT])
        m.snapshot()
        t_snap = m.get_time()
        assert t_snap == T0 + 360.0 + DT
        its1 = m.run([DT, DT, DT])
        s1, t1 = state(m), m.get_time()
        m.rollback()
        assert m.get_time() == t_snap
        its2 = m.run([DT, DT, DT])
        assert list(its1) == list(its2) and m.get_time() == t1
        for x, y in zip(s1, state(m)):
            assert np.array_equal(x, y)
    finally:
        m.close()


def test_budget_records_close_and_count_the_moulins():
    c = make_case(seed=7)
    mo = moulin_set(c[0].shape[0], c[3])
    dts = ShaktiOracle.dt_schedule(np.linspace(0, 6 * DT, 7))[:6]
    m, plain = make_model(*c), make_model(*c)
    o = moulin_oracle(c, mo, T0)
    try:
        set_moulins(m, mo)
        m.set_time(T0)
        m.record_diagnostics(len(dts))
        t = T0
        for dt in dts:
            m.newton_solve(dt)
            shot = m.diagnostics(dt)                         # one-shot record of the converged state
            for k in ("N", "N_n", "b", "melt_n"):
                getattr(o, k)[:] = m.get_field(k)
            o.q[:] = m.get_flux()
            o.t = t
            errs = record_errors(shot, moulin_diagnostics(o, dt), CM)
            assert not {k: v for k, v in errs.items() if v > (0.0 if k in ("N_min", "N_max", "b_max") else 1e-12)}, errs
            m.update_q_melt()
            m.update_b(dt)
            m.copy_N_to_N_n()
            t += dt
        rows = m.read_diagnostics()
        assert rows.shape == (len(dts), len(capi.DIAGNOSTICS))
        base_input = plain.diagnostics(DT)["input"]             # int inputs (does not depend on the state)
        t = T0
        for row, dt in zip(rows, dts):
            r = dict(zip(capi.DIAGNOSTICS, row))
            qsum = m.moulin_discharge(t + dt).sum()
            t += dt
            assert qsum > 0 and r["input"] == pytest.approx(base_input + qsum, rel=1e-13)
            scale = abs(r["input"]) + CM * abs(r["melt"]) + abs(r["closure"]) + abs(r["storage"]) + abs(r["outflow"])
            rhs = r["input"] - CM * r["melt"] + r["closure"] + r["storage"] + r["imbalance"]
            assert abs(r["outflow"] - rhs) <= 1e-10 * scale, r
            assert abs(r["imbalance"]) <= np.sqrt(c[0].shape[0]) * r["residual"] + 1e-12 * scale, r
    finally:
        m.close()
        plain.close()


def test_removed_moulins_launch_nothing_and_change_nothing():
    c = make_case(seed=8)
    mo = moulin_set(c[0].shape[0], c[3])
    never, zeroed = make_model(*c), make_model(*c)
    try:
        set_moulins(zeroed, mo)
        zeroed.set_moulins([], [], [])
        per_step = []
        for m in (never, zeroed):
            counts = [m.stats()["kernel_launches"]]
            for dt in (360.0, DT, DT):
                m.step(dt)
                counts.append(m.stats()["kernel_launches"])
            per_step.append(np.diff(counts))
        assert np.array_equal(per_step[0], per_step[1])
        for x, y in zip(state(never), state(zeroed)):
            assert np.array_equal(x, y)
    finally:
        never.close()
        zeroed.close()


def test_invalid_arguments_are_refused_and_leave_the_model_usable():
    c = make_case(seed=9)
    nv, bc = c[0].shape[0], c[3]
    mo = moulin_set(nv, bc)
    m = make_model(*c)
    try:
        set_moulins(m, mo)
        m.set_time(T0)
        F0 = m.assemble(DT)[0]
        tk, qk = np.array([0.0, 10.0, 20.0]), np.array([1.0, 2.0, 3.0])
        free = mo[0][0]
        bad = [
            dict(vertex=[-1], times=[tk], discharges=[qk]),
            dict(vertex=[nv], times=[tk], discharges=[qk]),
            dict(vertex=[int(bc[0])], times=[tk], discharges=[qk]),                    # Dirichlet dof
            dict(vertex=[free, free], times=[tk, []], discharges=[qk, []]),             # empty hydrograph
            dict(vertex=[free], times=[[0.0, 10.0, 10.0]], discharges=[qk]),           # repeated knot time
            dict(vertex=[free], times=[[0.0, 20.0, 10.0]], discharges=[qk]),           # decreasing
            dict(vertex=[free], times=[[0.0, np.nan, 20.0]], discharges=[qk]),
            dict(vertex=[free], times=[tk], discharges=[[1.0, np.inf, 3.0]]),
            dict(vertex=[free], times=[[-np.inf, 0.0, 1.0]], discharges=[qk]),
            dict(vertex=[free], times=[tk], discharges=[qk], period=-1.0),
            dict(vertex=[free], times=[tk], discharges=[qk], period=np.nan),
            dict(vertex=[free], times=[tk], discharges=[qk], period=np.inf),
        ]
        for kw in bad:
            with pytest.raises(capi.ShaktiError) as e:
                m.set_moulins(**kw)
            assert e.value.code == -1, kw
        for t in (np.nan, np.inf):
            with pytest.raises(capi.ShaktiError) as e:
                m.set_time(t)
            assert e.value.code == -1
        # a Dirichlet set that would put a moulin on a Dirichlet dof
        with pytest.raises(capi.ShaktiError) as e:
            m.set_dirichlet(np.append(bc, free), c[4])
        assert e.value.code == -1 and "moulin" in str(e.value)
        # nothing changed: the same residual, the same time, and the model still steps
        assert m.get_time() == T0
        assert np.array_equal(m.assemble(DT)[0], F0)
        it, conv = m.step(DT)
        assert conv and it >= 1 and m.get_time() == T0 + DT
    finally:
        m.close()


def test_solve_md_setup_moulins_like_matches_reference(tmp_path):
    """solvers.solve(md) with md.moulins (x, y, times, Q) on a small setup_moulins_like case, time axis starting at
    5 h: the saved fields equal a reference run stepped with o.t = timesteps[i] - dt_i (step 0 forced at 5 h, not at
    0.5 h), and the model's clock and step counter end at the last time step."""
    import solvers
    from _synthetic import md_from_case
    from scipy.spatial import cKDTree
    from shakti_b200 import fem
    nt = 8
    case = configs.moulins_like(nx=50, ny=10, nsteps=nt)
    case.timesteps = case.timesteps + 5 * 3600.0
    md = md_from_case(fem.comm_world(), case, str(ROOT / "shakti-fenics_b200" / "setups" / "setup_moulins_like.py"),
                      nt_save=2, nt_check=4, results_name=str(tmp_path / "run"), solver_options=dict(linear_rtol=1e-13))
    md.moulins = case.meta["moulins"]
    md.moulin_period = case.meta["moulin_period"]
    solvers.solve(md)
    out = Path(md.results_name)
    N, b = np.load(out / "N.npy"), np.load(out / "b.npy")
    model = md.solver.model
    assert model.stats()["steps"] == nt and model.get_time() == pytest.approx(md.timesteps[-1], rel=1e-15)
    bc = solvers.get_bcs(md)[0].dofs
    tree = cKDTree(case.xy)
    mo = [(int(tree.query([x, y])[1]), t, q) for x, y, t, q in md.moulins]
    f = case.fields
    o = moulin_oracle((case.xy, case.cells, f, bc, case.N_bdry), mo, 0.0)
    j = 0
    for i, dt in enumerate(o.dt_schedule(md.timesteps)):
        o.t = md.timesteps[i] - dt
        o.step(dt)
        if i % md.nt_save == 0:
            assert relinf(N[j], o.N) < 1e-8, (i, relinf(N[j], o.N))
            assert relinf(b[j], o.b) < 1e-8, (i, relinf(b[j], o.b))
            j += 1
    assert j == nt // md.nt_save
    assert relinf(md.final["N"].x.array, o.N) < 1e-8


@pytest.mark.parametrize("p2p", ["1", "0"], ids=["p2p-kernels", "nccl-only"])
def test_multi_gpu_moulins(p2p):
    """2 GPUs (skipped when fewer are visible), launched by torchrun: tests/multi_gpu_moulin_check.py."""
    import os
    import subprocess
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    script = Path(__file__).with_name("multi_gpu_moulin_check.py")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29531" if p2p == "1" else "29533", str(script)],
                       capture_output=True, text=True, timeout=900, env={**os.environ, "SHAKTI_P2P": p2p})
    assert "MULTI_GPU_MOULINS PASSED" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]
