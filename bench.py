#!/usr/bin/env python
"""Headline benchmark: SHAKTI transient time-steps/s at 16M dofs (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            # the B200 path (this repo)
  python bench.py --impl reference --gpus N --steps K ...  # CPU arm: the oracle port on host cores
  python bench.py --scaling weak --gpus N ...              # C5: 8M dofs per GPU, lake fill-drain pulse
  python bench.py ... --dump-outputs DIR                   # also write the last timed step's outputs as DIR/*.npy

A "step" is one pass of reference source/solvers.py:179-229 (Newton solve for N with F+J
assembly and the Krylov/AMG linear solves, then the q / melt_n / b nodal updates) on the
synthetic config C4 of SURVEY.md §8d (4000 x 4000 vertices, jittered margin mesh, turbulent
K(b,Re)); N > 1 partitions that same mesh over N GPUs (strong scaling).  With --scaling weak the
mesh grows with N (C5: lakes with storage, time-dependent inputs uploaded every step).  One JSON
line is printed by rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
for _p in (str(ROOT), str(ROOT / "shakti-fenics_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

METRIC = "time_steps_per_sec_at_16M_dofs"
UNIT = "steps/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="strong: C4 (16M dofs) partitioned over N GPUs; weak: C5, 8M dofs per GPU")
    ap.add_argument("--nside", type=int, default=None, help="vertices per side (default 4000 -> 16M dofs; weak: sqrt(8e6 N))")
    ap.add_argument("--precond", default="amg")
    ap.add_argument("--linear-rtol", type=float, default=1e-12)
    ap.add_argument("--amg-refresh-every", type=int, default=None, help="override shakti_options.amg_refresh_every")
    ap.add_argument("--amg-replicate-below", type=int, default=None)
    ap.add_argument("--lagged-smoother-halo", action="store_true", help="multi-GPU: amg_smoother_halo = 0")
    ap.add_argument("--linear-forcing", type=float, default=None, help="override shakti_options.linear_forcing (0 = fixed tolerance)")
    ap.add_argument("--no-graph", action="store_true", help="do not replay the AMG V-cycle as a CUDA graph")
    ap.add_argument("--cpu-sample-nside", type=int, default=None,
                    help="mesh side of the bounded CPU sample (default: sized so that the CPU run takes ~2 minutes)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-variant", default="both", choices=["both", "h2d", "d2h", "none"],
                    help="diagnostic: which host copies the end-to-end leg performs")
    ap.add_argument("--no-kernels", action="store_true", help="skip the per-kernel roofline timings")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one left to the caller as DIR/<name>.npy (float64): "
                         "the fields N, b, qx, qy, melt_n (on meshes above 2^20 vertices the same seeded sample of 2^20 "
                         "vertices in every run) and the Newton iterations of the timed steps")
    return ap.parse_args()


def peaks():
    f = ROOT / "MEASURED_PEAKS.json"
    if f.exists():
        return float(json.loads(f.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------ CPU arm
def _oracle_backend():
    """The CPU arm runs the oracle's compiled element kernels (oracle/shakti_oracle_c.c, OpenMP over cells -- the
    reference's element kernels are FFCx-generated C as well) when `make -C oracle` has built them, with the
    fill-reducing MMD(A'+A) ordering for SuperLU; otherwise the numpy restatement.  Both are the same algorithm
    (tests/test_oracle.py: 1e-13)."""
    from oracle import cbackend
    try:
        if cbackend.available():
            return (dict(backend="c", permc_spec="MMD_AT_PLUS_A"), cbackend.threads(),
                    "C element kernels (OpenMP) + scipy SuperLU, MMD(A'+A) ordering")
    except OSError as e:                      # library built for another host: say so and time the numpy form
        print(f"[bench] oracle C backend not loadable ({e}); CPU arm uses the numpy oracle", file=sys.stderr)
    return {}, cpu_threads(), "numpy element kernels + scipy SuperLU"


def _oracle_for(case):
    from oracle.shakti_oracle import ShaktiOracle
    o = ShaktiOracle(case.xy, case.cells, **_oracle_backend()[0])
    for k in ("z_b", "z_s", "G", "inputs", "storage", "b", "N_n", "melt_n"):
        getattr(o, k)[:] = case.fields[k]
    o.q[:] = case.fields["q"]
    o.set_dirichlet(case.bc_dofs, case.N_bdry)
    o.start()
    return o


def cpu_threads():
    """numpy/scipy threads the CPU restatement can use here (BLAS pools; SuperLU itself is serial)."""
    try:
        from threadpoolctl import threadpool_info
        n = max([p.get("num_threads", 1) for p in threadpool_info()] or [1])
    except Exception:
        n = 1
    return int(n)


def cpu_sample_nside(requested, n_steps, budget_s=90.0):
    """Bounded CPU sample: the mesh side whose `n_steps` oracle steps (the first one from the initial state:
    ~10 Newton iterations instead of 3) take about `budget_s` seconds.  Cost model measured with the compiled
    element kernels + SuperLU/MMD on the build container's cores: (30 + 0.07 sqrt(dofs)) us per dof and step
    (39 us at 40k dofs, 72 us at 490k, 101 us at 1M: the sparse LU is super-linear)."""
    if requested:
        return requested
    per_step = budget_s / (max(n_steps, 1) - 1 + 3.3)
    lo, hi = 1.0e4, 1.0e6
    for _ in range(40):
        d = 0.5 * (lo + hi)
        if d * 1e-6 * (30.0 + 0.07 * d ** 0.5) > per_step:
            hi = d
        else:
            lo = d
    return int(min(1000, max(100, lo ** 0.5)))


def cpu_oracle_rate(nside, steps, warmup, target_dofs):
    """Time the CPU oracle (numpy assembly + SuperLU, the stand-in for FEniCSx/PETSc LU) on a bounded
    sample: the same C4 fields on an nside x nside sub-size mesh.  Returns steps/s EXTRAPOLATED linearly in
    dofs to the target size (optimistic for the CPU: sparse LU is super-linear), the raw steps/s on the
    sample and a description."""
    from shakti_b200 import configs
    case = configs.dofs16m(nside=nside, nsteps=max(steps + warmup + 1, 4))
    o = _oracle_for(case)
    dts = case.dts(steps + warmup)
    for dt in dts[:warmup]:
        o.step(dt)
    t0, c0 = time.perf_counter(), time.process_time()
    its = [o.step(dt)[0] for dt in dts[warmup:]]
    el, cpu = time.perf_counter() - t0, time.process_time() - c0
    raw = steps / el
    scaled = raw * (case.n_vert / float(target_dofs))
    _, thr, what = _oracle_backend()
    sample = (f"{steps} oracle steps ({what}; {thr} threads for the element loops, the sparse LU itself is serial; measured CPU time / wall "
              f"time = {cpu / el:.1f} cores busy) on a {nside}x{nside}-vertex C4 mesh "
              f"({case.n_vert} dofs, {np.mean(its):.1f} Newton its/step): {raw:.4g} steps/s measured; `value` is that rate "
              f"EXTRAPOLATED by the dofs ratio {case.n_vert}/{target_dofs} (linear, optimistic for LU)")
    return scaled, raw, sample, el


def same_config_c2(cpu_steps=2, gpu_steps=20):
    """CPU oracle and the B200 path on the SAME config, unscaled: C2 (rectangle, 250k P1 triangles, steady
    melt forcing; BASELINE.json configs[1]).  The two warm-up steps (the 360 s first step with its ~10 Newton
    iterations would cost the CPU over a minute) run on the GPU; its state is handed to the oracle, both then
    take the same `cpu_steps` steps (fields compared), and the GPU is timed over `gpu_steps` more.
    -> dict(config, cpu_steps_s, gpu_steps_s, ratio, ...)."""
    from shakti_b200 import capi, configs
    case = configs.rect_steady(nsteps=cpu_steps + gpu_steps + 8)
    dts = case.dts()
    out = {"config": f"C2 rectangle 100x50 km, {case.cells.shape[0]} P1 triangles, {case.n_vert} dofs, steady melt forcing; "
                     "state after 2 warm-up steps (run on the GPU) given to both"}
    m = capi.Model(case.xy, case.cells)
    configs.apply_case(m, case)
    m.run(dts[:2])
    o = _oracle_for(case)
    for k in ("b", "N_n", "melt_n"):
        getattr(o, k)[:] = m.get_field(k)
    o.q[:] = m.get_flux()
    o.start()
    t0 = time.perf_counter()
    its = [o.step(dt)[0] for dt in dts[2:2 + cpu_steps]]
    out["cpu_steps_s"] = cpu_steps / (time.perf_counter() - t0)
    out["cpu_steps"] = cpu_steps
    out["cpu_threads"] = _oracle_backend()[1]
    out["cpu_impl"] = _oracle_backend()[2]
    out["cpu_newton_its"] = [int(i) for i in its]
    its_g = m.run(dts[2:2 + cpu_steps])
    out["gpu_newton_its"] = [int(i) for i in its_g]
    out["N_rel_err_gpu_vs_cpu"] = float(np.max(np.abs(m.get_field("N") - o.N)) / np.max(np.abs(o.N)))
    out["b_rel_err_gpu_vs_cpu"] = float(np.max(np.abs(m.get_field("b") - o.b)) / np.max(np.abs(o.b)))
    _, ms = m.run_timed(dts[2 + cpu_steps:2 + cpu_steps + gpu_steps])
    out["gpu_steps_s"] = gpu_steps / (ms / 1e3)
    out["gpu_steps"] = gpu_steps
    out["ratio"] = out["gpu_steps_s"] / out["cpu_steps_s"]
    m.close()
    return out


def run_reference(args):
    """--impl reference: the reference's algorithm on the host CPU (oracle port: FEniCSx/PETSc are not
    installable here, see DESIGN.md).  Rank 0 only.  The 16M-dof LU neither fits nor finishes, so every
    step is a bounded sample (same fields, smaller mesh) and `value` is an extrapolation, flagged as such;
    the unscaled same-config comparison (C2) is part of the B200 arm's cpu_baseline."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # torchrun gives every rank OMP_NUM_THREADS=1; here the other ranks have just exited, so rank 0 may use the
    # whole host (the OpenMP runtime of the oracle's C kernels reads the variable when the library is loaded, below)
    if int(os.environ.get("WORLD_SIZE", "1")) > 1 and os.environ.get("OMP_NUM_THREADS") == "1":
        os.environ["OMP_NUM_THREADS"] = str(os.cpu_count() or 1)
    nside = args.nside or 4000
    target = nside * nside
    nside_cpu = cpu_sample_nside(args.cpu_sample_nside, args.steps + 1)
    scaled, raw, sample, el = cpu_oracle_rate(nside_cpu, args.steps, min(args.warmup, 1), target)
    threads = _oracle_backend()[1]
    line = {
        "impl": "reference", "metric": METRIC, "value": scaled, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": min(args.warmup, 1), "ms_per_step": 1e3 / scaled, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic", "extrapolated": True, "same_config": False,
        "config": {"workload": f"C4 synthetic ice-sheet margin mesh {nside}x{nside} vertices ({target} dofs), "
                               "turbulent K(b,Re), dt=3600 s", "sample_nside": nside_cpu,
                   "sample_seconds": el, "raw_steps_per_sec_on_sample": raw},
        "cpu_baseline": {"value": scaled, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                         "raw_steps_per_sec_on_sample": raw, "extrapolated": True},
        "e2e": {"value": scaled, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------ B200 arm
DUMP_SAMPLE = 1 << 20          # vertices per dumped field: five float64 fields stay at 40 MB


def dump_outputs(m, its, out_dir, dist, rank):
    """--dump-outputs: the state the timed steps hand back to their caller (N, b, q, melt_n) and their Newton
    iteration counts, so that two builds run with the same arguments can be compared output for output."""
    import torch
    n = m.n_vert
    idx = np.arange(n) if n <= DUMP_SAMPLE else np.sort(np.random.default_rng(0).choice(n, DUMP_SAMPLE, replace=False))
    q = m.get_flux()
    out = {k: m.get_field(k)[idx] for k in ("N", "b", "melt_n")}
    out["qx"], out["qy"] = q[idx, 0], q[idx, 1]
    if dist is not None:           # each rank returns its owned vertices and zeros elsewhere
        for k, v in out.items():
            t = torch.from_numpy(np.ascontiguousarray(v)).cuda()
            dist.all_reduce(t)
            out[k] = t.cpu().numpy()
    out["newton_its"] = np.asarray(its, dtype=np.float64)
    if rank == 0:
        os.makedirs(out_dir, exist_ok=True)
        for k, v in out.items():
            np.save(os.path.join(out_dir, f"{k}.npy"), np.asarray(v, dtype=np.float64))


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
        return
    import torch
    from shakti_b200 import capi, configs

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the B200 path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            uid = torch.tensor(list(capi.comm_unique_id()), dtype=torch.uint8, device="cuda")
        dist.broadcast(uid, 0)
        capi.comm_init(bytes(uid.cpu().tolist()), rank, world, local_rank)
    assert args.gpus == world, f"--gpus {args.gpus} but WORLD_SIZE={world}"

    weak = args.scaling == "weak"
    t_setup = time.perf_counter()
    nsteps_total = args.warmup + 2 * args.steps + 4
    if weak:
        nside = args.nside or int(round((8.0e6 * world) ** 0.5))
        case = configs.lakes_fill_drain(nside=nside, nsteps=nsteps_total)
        # the pulse is centred in the benchmark window so that the forcing really changes from step to step
        case.meta["t_pulse"], case.meta["tau"] = 0.5 * nsteps_total * 3600.0, 0.25 * nsteps_total * 3600.0
    else:
        nside = args.nside or 4000
        case = configs.dofs16m(nside=nside, nsteps=nsteps_total)
    nv = case.n_vert
    extra = {} if args.amg_refresh_every is None else {"amg_refresh_every": args.amg_refresh_every}
    if args.amg_replicate_below is not None:
        extra["amg_replicate_below"] = args.amg_replicate_below
    if args.linear_forcing is not None:
        extra["linear_forcing"] = args.linear_forcing
    if args.no_graph:
        extra["amg_cuda_graph"] = 0
    if args.lagged_smoother_halo:
        extra["amg_smoother_halo"] = 0
    m = capi.Model(case.xy, case.cells, device=local_rank, precond=args.precond, linear_rtol=args.linear_rtol, **extra)
    configs.apply_case(m, case)
    dts = case.dts()
    owned = m.owned()
    n_own = int(owned.size)
    setup_s = time.perf_counter() - t_setup

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def maxr(x):
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # pinned host buffers of the end-to-end path: this rank's owned slice (the caller places it with the
    # index map of shakti_get_owned), two output sets for double buffering
    h_in = capi.PinnedArray(n_own)
    out_sets = [[capi.PinnedArray(n_own) for _ in range(4)] for _ in range(2)]

    def inputs_at(step_index):
        if weak:
            return configs.lake_pulse_inputs(case, case.timesteps[step_index])[owned]
        return case.fields["inputs"][owned]

    # ---- warm-up (untimed)
    if weak:
        its_w = []
        for i in range(args.warmup):
            h_in.array[:] = inputs_at(i)
            its_w.append(m.step_host_async(dts[i], h_in.array.ctypes.data, owned_only=True)[0])
    else:
        its_w = m.run(dts[: args.warmup])
    m.snapshot()              # the end-to-end leg repeats exactly the timed steps from this state
    st0 = m.stats()
    # ---- timed region: exactly K steps, max over ranks
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    barrier()
    if weak:
        # time-dependent forcing: every step uploads its inputs (pinned host -> device) before it runs; the K steps
        # are bracketed by a device synchronisation on both sides (every step ends with the host reading ||F||)
        pinned_t = [capi.PinnedArray(n_own) for _ in range(args.steps)]
        for i, pa in enumerate(pinned_t):
            pa.array[:] = inputs_at(args.warmup + i)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        its = []
        for i in range(args.steps):
            its.append(m.step_host_async(dts[args.warmup + i], pinned_t[i].array.ctypes.data, owned_only=True)[0])
        torch.cuda.synchronize()
        ms = 1e3 * (time.perf_counter() - t0)
    else:
        # device time (CUDA events on the library stream around exactly K steps)
        its, ms = m.run_timed(dts[args.warmup: args.warmup + args.steps])
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    ms = maxr(ms)
    st1 = m.stats()
    if args.dump_outputs:
        dump_outputs(m, its, args.dump_outputs, dist, rank)
    value = args.steps / (ms / 1e3)
    launches = st1["kernel_launches"] - st0["kernel_launches"]

    # ---- end-to-end: host buffers in the call; every step the forcing goes host -> device and b, N, qx, qy
    # come back into pinned host memory (nt_save = 1).  The copies of step k overlap step k+1
    # (shakti_step_host_async, two buffer sets); the timed region ends after the LAST copy has landed.
    e2e = None
    if not args.no_e2e:
        # same steps as the timed region (the transient gets harder as it develops: later steps need more Krylov
        # iterations, so the two rates are only comparable over the same step indices)
        # one untimed end-to-end step first: the staging buffers of the output path are allocated and the copy
        # stream is used for the first time outside the timed region (warm-up, like the W steps above)
        h_in.array[:] = inputs_at(args.warmup + args.steps)
        m.step_host_async(dts[args.warmup + args.steps], h_in.array.ctypes.data, *[b.array.ctypes.data for b in out_sets[0]],
                          owned_only=True)
        m.wait_outputs()
        m.rollback()
        k0 = args.warmup
        # the step's inputs already sit in pinned host memory when the step is called (filling that memory is
        # the caller's data production, not the path being measured): one array in strong mode (static
        # forcing), one per step in weak mode (time-dependent forcing)
        if weak:
            pinned_in = [capi.PinnedArray(n_own) for _ in range(args.steps)]
            for i, pa in enumerate(pinned_in):
                pa.array[:] = inputs_at(k0 + i)
        else:
            h_in.array[:] = inputs_at(k0)
            pinned_in = [h_in] * args.steps
        barrier()
        t0 = time.perf_counter()
        chk = 0.0
        use_in, use_out = args.e2e_variant in ("both", "h2d"), args.e2e_variant in ("both", "d2h")
        for i in range(args.steps):
            bufs = out_sets[i % 2]
            m.step_host_async(dts[k0 + i], pinned_in[i].array.ctypes.data if use_in else None,
                              *([b.array.ctypes.data for b in bufs] if use_out else [None] * 4), owned_only=True)
            if i >= 1:                       # read the PREVIOUS step's result on the host while this one's copies fly
                chk += float(out_sets[(i - 1) % 2][1].array[0])
        m.wait_outputs()
        chk += float(out_sets[(args.steps - 1) % 2][1].array[0])
        barrier()
        el = maxr(time.perf_counter() - t0)
        e2e = {"value": args.steps / el, "unit": UNIT, "h2d_bytes_per_step": 8 * nv, "d2h_bytes_per_step": 4 * 8 * nv,
               "how": "shakti_step_host_async: per step the forcing H2D and b,N,qx,qy D2H (nt_save=1) through pinned host "
                      "buffers, every rank moving its owned slice; D2H double-buffered behind the next step; wall clock incl. "
                      "the last copy, max over ranks", "checksum": chk, "variant": args.e2e_variant,
               "its_e2e": (m.stats()["linear_its"] - st1["linear_its"]) / args.steps}

    # ---- rooflines, live CUDA events on the library stream.  Dominant kernel of the step (largest share
    # in profiles/r2_launch_shares_*.csv): the AMG smoother amg_cheby_kernel on the fine level.
    peak, peak_src = peaks()
    kern, roofline = {}, None
    if not args.no_kernels:
        for k in ("spmv", "assemble", "kbar", "nodal", "dot", "axpy"):
            t_ms = m.time_kernel(k, reps=20, dt=3600.0)
            by = m.kernel_bytes(k)
            kern[k] = {"ms": t_ms, "algorithmic_GB": by / 1e9, "GBps": by / 1e9 / (t_ms / 1e3), "frac": by / 1e9 / (t_ms / 1e3) / peak}
        kern["kbar"]["bound"] = "fp64 pipe (16 x (sqrt + div) per cell, once per step): the HBM fraction is not its roofline"
        kern["nodal"]["what"] = "update_q_melt_kernel + update_b_kernel, bytes 12 Ne + 104 Nv (SURVEY 8d, single-pass ideal)"
        levels = []
        if args.precond == "amg":
            for lvl in range(st1["amg_levels"]):
                try:
                    r = m.time_amg_smoother(lvl, reps=20)
                except capi.ShaktiError:
                    break
                if r["rows"] == 0:
                    continue
                gbs = r["bytes"] / 1e9 / (r["ms"] / 1e3)
                levels.append({"level": lvl, "rows": r["rows"], "nnz": r["nnz"], "value_bytes": r["value_bytes"], "us": 1e3 * r["ms"],
                               "algorithmic_GB": r["bytes"] / 1e9,
                               "GBps": gbs, "frac": gbs / peak})
        traffic = None
        tf = ROOT / "profiles" / "r2_traffic.json"
        if tf.exists() and world == 1 and not weak:
            t_all = json.loads(tf.read_text())
            t_ = t_all.get("amg_cheby_fine_fp32") or t_all.get("amg_cheby_fine", {})
            # the capture is of the fp32 level copy: not valid for the opt-in half-precision smoother
            if t_.get("nside") == nside and levels and levels[0]["value_bytes"] == 4:
                traffic = t_["traffic_bytes"]       # dram read+write per launch, ncu --set full (profiles/)
        if levels:
            l0 = levels[0]
            kname = ("amg_cheby_h_kernel (AMG smoother, fine level, half-precision row-scaled SELL-32 copy of J, fp32 vectors)"
                     if l0["value_bytes"] == 2 else "amg_cheby_kernel<float,1> (AMG smoother, fine level, fp32 SELL-32 copy of J)")
            roofline = {"bound": "hbm", "kernel": kname,
                        "achieved": l0["GBps"], "peak": peak, "unit": "GB/s", "frac": l0["frac"], "traffic": traffic,
                        "algorithmic_bytes": l0["algorithmic_GB"] * 1e9, "peak_source": peak_src, "levels": levels,
                        "how": "(value_bytes+4) nnz + 28 rows algorithmic bytes / mean of 20 launches, CUDA events on the library stream; "
                               "matrix >> L2; largest share of the step in profiles/r2_launch_shares_16M_one_step.csv",
                        "secondary": {"spmv_fine_fp64": kern["spmv"], "assemble_blocks": kern["assemble"]}}
        else:
            roofline = {"bound": "hbm", "kernel": "spmv_sell_kernel<0,double,1> (fine Jacobian, fp64 SELL-32)", "achieved": kern["spmv"]["GBps"],
                        "peak": peak, "unit": "GB/s", "frac": kern["spmv"]["frac"], "traffic": None,
                        "algorithmic_bytes": m.kernel_bytes("spmv"), "peak_source": peak_src}

    if rank != 0:
        m.close()
        if dist is not None:
            capi.comm_finalize()
            dist.destroy_process_group()
        return
    m.close()
    cpu_baseline = None
    if not args.no_cpu_baseline and world == 1 and not weak:
        scaled, raw, sample, _ = cpu_oracle_rate(cpu_sample_nside(args.cpu_sample_nside, 3), 2, 1, nv)
        cpu_baseline = {"value": scaled, "unit": UNIT, "cores": _oracle_backend()[1], "kind": "port", "sample": sample,
                        "raw_steps_per_sec_on_sample": raw, "extrapolated": True,
                        "same_config": same_config_c2()}
    n_newton = st1["newton_its"] - st0["newton_its"]
    n_krylov = st1["linear_its"] - st0["linear_its"]
    workload = (f"C5 lakes fill-drain, {nside}x{nside} vertices ({nv} dofs = {nv / world / 1e6:.2f} M per GPU), storage on, inputs(t) pulse "
                "uploaded every step, dt=3600 s" if weak else
                f"C4 synthetic ice-sheet margin mesh {nside}x{nside} vertices ({nv} dofs, {case.cells.shape[0]} P1 triangles), "
                "turbulent K(b,Re), dt=3600 s")
    line = {
        "metric": "time_steps_per_sec_weak_8M_dofs_per_gpu" if weak else METRIC, "value": value, "unit": UNIT, "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload,
                   "parallelism": f"mesh partition x{world}" if world > 1 else "single GPU",
                   "l2": "inputs larger than L2 (matrix + vectors >> 126 MB)",
                   "newton_its_per_step": n_newton / args.steps, "krylov_its_per_solve": n_krylov / max(n_newton, 1),
                   "linear_solver": "gmres", "precond": args.precond, "linear_rtol": args.linear_rtol,
                   "linear_forcing": float(m.options.linear_forcing),
                   "amg_levels": st1["amg_levels"], "amg_refreshes_in_timed_region": st1["amg_refreshes"] - st0["amg_refreshes"],
                   "amg_operator_complexity": st1["amg_operator_complexity"],
                   "setup_seconds": setup_s, "host_max_rss_gb": __import__("resource").getrusage(0).ru_maxrss / 1048576.0,
                   "warmup_newton_its": [int(v) for v in its_w],
                   "timed_newton_its": [int(v) for v in its]},
        "roofline": roofline, "kernels": kern, "cpu_baseline": cpu_baseline, "e2e": e2e, "gpu_launches": int(launches),
        "clocks": clocks,
    }
    print(json.dumps(line), flush=True)
    if dist is not None:
        capi.comm_finalize()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
