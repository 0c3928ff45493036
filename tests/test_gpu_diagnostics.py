"""Water-budget diagnostics on the GPU: the one-shot record against the CPU oracle at the same state, the records
taken during a run against one-shot records of the same states, the discrete budget identity at C2 size, that
recording off launches nothing, and the solvers.solve(md) path."""
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
for p in (ROOT / "shakti-fenics_b200" / "source", ROOT / "shakti-fenics_b200" / "setups"):
    if str(p) not in sys.path:
        sys.path.insert(0, str(p))

from common import make_case, make_model, make_oracle  # noqa: E402
from budget_reference import oracle_diagnostics  # noqa: E402
from multi_gpu_diagnostics_check import record_errors  # noqa: E402
from oracle.shakti_oracle import Params, ShaktiOracle  # noqa: E402
from shakti_b200 import capi  # noqa: E402

pytestmark = pytest.mark.gpu

DT = 3600.0
CM = 1 / 917 - 1 / 1000


def _assert_records_close(got, ref):
    errs = record_errors(got, ref, CM)
    bad = {k: v for k, v in errs.items() if v > (0.0 if k in ("N_min", "N_max", "b_max") else 1e-12)}
    assert not bad, (bad, got, ref)


@pytest.mark.parametrize("n", [3.0, 2.5], ids=["n3-radon7", "n2.5-table"])
@pytest.mark.parametrize("kernel", [0, 1], ids=["row-block-gather", "cell-atomics"])
def test_one_shot_matches_oracle(kernel, n):
    c = make_case(nx=40, ny=28, seed=11)
    o = make_oracle(*c, params=Params(n=n))
    p = capi.default_params()
    p.n = n
    m = make_model(*c, params=p, assembly_kernel=kernel)
    try:
        _assert_records_close(m.diagnostics(DT), oracle_diagnostics(o, DT))        # start state (N = N_n)
        m.newton_solve(DT)
        o.N[:] = m.get_field("N")                                           # the GPU's converged state
        d = m.diagnostics(DT)
        _assert_records_close(d, oracle_diagnostics(o, DT))
        assert d["N_min"] < d["N_mean"] < d["N_max"] and d["outflow"] != 0 and d["storage"] != 0
    finally:
        m.close()


def test_one_shot_matches_oracle_negative_gap_start():
    c = make_case(seed=4, neg_b=True, turbulent=False)
    o = make_oracle(*c)
    m = make_model(*c)
    try:
        _assert_records_close(m.diagnostics(360.0), oracle_diagnostics(o, 360.0))
    finally:
        m.close()


def test_records_of_a_run_equal_one_shot_records():
    """shakti_run with recording on vs a twin model driven step by step with a one-shot record taken after each
    Newton solve (the state a record describes): columns 3-14 bitwise, 0-2 = dt, Newton count, final residual."""
    c = make_case(seed=2)
    dts = ShaktiOracle.dt_schedule(np.linspace(0, 8 * DT, 9))[:6]
    a, b = make_model(*c), make_model(*c)
    try:
        a.record_diagnostics(6)
        its = a.run(dts)
        rows = a.read_diagnostics()
        assert rows.shape == (6, len(capi.DIAGNOSTICS))
        assert rows[-1, 2] == a.stats()["last_residual"]
        for i, dt in enumerate(dts):
            it, _ = b.newton_solve(dt)
            res = b.stats()["last_residual"]
            shot = b.diagnostics(dt)
            b.update_q_melt()
            b.update_b(dt)
            b.copy_N_to_N_n()
            assert it == its[i]
            assert rows[i, 0] == dt and rows[i, 1] == its[i] and rows[i, 2] == res
            assert np.array_equal(rows[i, 3:], [shot[k] for k in capi.DIAGNOSTICS[3:]]), i
        assert a.read_diagnostics().shape == (0, len(capi.DIAGNOSTICS))   # reading empties the buffer
    finally:
        a.close()
        b.close()


def test_budget_identity_at_c2_size():
    """C2 (250k triangles): every converged step closes the budget to 1e-10 of its scale, and the imbalance is the
    sum of the assembled residual over the non-Dirichlet rows (the lifting term is zero: N = N_bdry exactly on the
    Dirichlet rows once Newton has taken a step)."""
    from shakti_b200 import configs
    case = configs.rect_steady(nsteps=4)
    m = configs.apply_case(capi.Model(case.xy, case.cells), case)
    try:
        m.record_diagnostics(3)
        m.run(case.dts(3))
        rows = m.read_diagnostics()
        it, _ = m.newton_solve(DT)
        F, N = m.get_field("residual"), m.get_field("N")
        d = m.diagnostics(DT)
        isbc = np.zeros(case.n_vert, dtype=bool)
        isbc[case.bc_dofs] = True
        assert it >= 1 and np.all(N[isbc] == case.N_bdry)
        for r in list(rows) + [[d[k] for k in capi.DIAGNOSTICS]]:
            r = dict(zip(capi.DIAGNOSTICS, r))
            scale = abs(r["input"]) + CM * abs(r["melt"]) + abs(r["closure"]) + abs(r["storage"]) + abs(r["outflow"])
            rhs = r["input"] - CM * r["melt"] + r["closure"] + r["storage"] + r["imbalance"]
            assert abs(r["outflow"] - rhs) <= 1e-10 * scale, r
            assert abs(r["imbalance"]) <= np.sqrt(case.n_vert) * r["residual"] + 1e-12 * scale
            assert r["outflow"] > 0 and r["area"] == pytest.approx(5e9, rel=1e-12)
        assert abs(d["imbalance"] - F[~isbc].sum()) <= 1e-10 * (abs(d["input"]) + abs(d["outflow"]))
    finally:
        m.close()


def test_recording_off_launches_nothing_full_buffer_and_rollback():
    c = make_case(seed=3)
    never, zeroed, rec = make_model(*c), make_model(*c), make_model(*c)
    try:
        zeroed.record_diagnostics(4)
        zeroed.record_diagnostics(0)
        per_step = []
        for m in (never, zeroed):
            counts = [m.stats()["kernel_launches"]]
            for dt in (360.0, DT, DT):
                m.step(dt)
                counts.append(m.stats()["kernel_launches"])
            per_step.append(np.diff(counts))
        assert np.array_equal(per_step[0], per_step[1])
        # a full buffer fails before the solve changes anything
        rec.record_diagnostics(1)
        rec.step(360.0)
        N0, b0, steps0 = rec.get_field("N"), rec.get_field("b"), rec.stats()["steps"]
        with pytest.raises(capi.ShaktiError) as e:
            rec.step(DT)
        assert e.value.code == -1 and "shakti_read_diagnostics" in str(e.value)
        with pytest.raises(capi.ShaktiError):
            rec.run([DT])
        assert np.array_equal(rec.get_field("N"), N0) and np.array_equal(rec.get_field("b"), b0)
        assert rec.stats()["steps"] == steps0
        assert rec.read_diagnostics().shape[0] == 1
        # rollback drops the rows recorded after the snapshot
        rec.record_diagnostics(4)
        rec.step(DT)
        rec.snapshot()
        rec.run([DT, DT])
        rec.rollback()
        rows = rec.read_diagnostics()
        assert rows.shape[0] == 1
        rec.run([DT, DT, DT])
        assert rec.read_diagnostics().shape[0] == 3
    finally:
        for m in (never, zeroed, rec):
            m.close()


def _md(tmp_path, name, nsteps, diagnostics_on, resume=False):
    from _synthetic import md_from_case
    from shakti_b200 import configs, fem
    case = configs.rect_steady(nx=60, ny=40, nsteps=8)
    md = md_from_case(fem.comm_world(), case, str(ROOT / "shakti-fenics_b200" / "setups" / "setup_rect250k.py"),
                      nt_save=2, nt_check=4, results_name=str(tmp_path / name))
    md.timesteps = case.timesteps[:nsteps]
    md.diagnostics_on = diagnostics_on
    md.resume = resume
    return md, case


def test_solve_md_writes_diagnostics_and_leaves_outputs_unchanged(tmp_path):
    import solvers
    nt = 8
    md, case = _md(tmp_path, "on", nt, True)
    solvers.solve(md)
    md_off, _ = _md(tmp_path, "off", nt, False)
    solvers.solve(md_off)
    on, off = Path(md.results_name), Path(md_off.results_name)
    assert not (off / "diagnostics.npz").exists()
    for f in ("b.npy", "N.npy", "qx.npy", "qy.npy"):
        assert (on / f).read_bytes() == (off / f).read_bytes(), f
    d = np.load(on / "diagnostics.npz")
    assert set(d.files) == {"t", *capi.DIAGNOSTICS}
    assert np.array_equal(d["t"], md.timesteps) and d["dt"].shape == (nt,)
    # the same steps driven by hand, with a one-shot record after each Newton solve
    from shakti_b200 import configs
    m = configs.apply_case(capi.Model(case.xy, case.cells, b_min=float(md.b_min)), case)
    try:
        m.set_dirichlet(solvers.get_bcs(md)[0].dofs, md.N_bdry)
        m.start()
        for i, dt in enumerate(case.dts(nt)):
            it, _ = m.newton_solve(dt)
            shot = m.diagnostics(dt)
            m.update_q_melt()
            m.update_b(dt)
            m.copy_N_to_N_n()
            assert d["newton_its"][i] == it and d["dt"][i] == dt
            for k in capi.DIAGNOSTICS[3:]:
                assert d[k][i] == pytest.approx(shot[k], rel=1e-9, abs=1e-9 * abs(shot["input"])), (i, k)
    finally:
        m.close()
    # a run stopped after 6 steps (last checkpoint after step 4) and resumed continues the same file
    md1, _ = _md(tmp_path, "resumed", 6, True, resume=True)
    solvers.solve(md1)
    assert np.load(Path(md1.results_name) / "diagnostics.npz")["t"].size == 6
    md2, _ = _md(tmp_path, "resumed", nt, True, resume=True)
    solvers.solve(md2)
    d2 = np.load(Path(md2.results_name) / "diagnostics.npz")
    assert np.array_equal(d2["t"], md.timesteps)
    for k in capi.DIAGNOSTICS[3:]:
        assert d2[k] == pytest.approx(d[k], rel=1e-8, abs=1e-8 * np.abs(d["input"]).max()), k


@pytest.mark.parametrize("p2p", ["1", "0"], ids=["p2p-kernels", "nccl-only"])
def test_multi_gpu_records_match_oracle(p2p):
    """2 GPUs (skipped when fewer are visible), launched by torchrun: tests/multi_gpu_diagnostics_check.py."""
    import os
    import subprocess
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    script = Path(__file__).with_name("multi_gpu_diagnostics_check.py")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29521" if p2p == "1" else "29523", str(script)],
                       capture_output=True, text=True, timeout=900, env={**os.environ, "SHAKTI_P2P": p2p})
    assert "MULTI_GPU_DIAGNOSTICS PASSED" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]
