"""Transient SHAKTI solver: same entry points as the reference (source/solvers.py:17-237)

    get_bcs(md) -> list            pde_solver(md, N, N_n, b, q, melt_n, storage, dt) -> solver
    solver.solve(N) -> (niter, converged)                                  solve(md) -> None

but everything the reference delegates to DOLFINx / FFCx / PETSc per time step runs in the
hand-written sm_100a CUDA library behind the C ABI (include/shakti_b200.h, bound by
shakti_b200.capi): P1 assembly of the residual and its N-Jacobian, the Newton loop, the
GMRES/AMG linear solves and the three nodal updates.  State stays resident in HBM; the host
only sees (niter, converged) each step and the four output fields every nt_save steps.
There is no CPU fallback: without the CUDA library or a B200 the calls raise.
"""
import os
import shutil
import sys
from pathlib import Path

import numpy as np

_PKG = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if _PKG not in sys.path:
    sys.path.insert(0, _PKG)

import params  # noqa: E402
from shakti_b200 import capi  # noqa: E402
from shakti_b200.fem import (Function, dirichletbc, locate_dofs_topological,  # noqa: E402
                             locate_entities_boundary)


class Constant:
    """dolfinx.fem.Constant stand-in: a scalar whose ``.value`` can be updated in place
    (the reference updates dt that way, solvers.py:82,176)."""

    def __init__(self, domain, value):
        self.value = float(value)


def get_bcs(md):
    # Dirichlet condition on effective pressure at the outflow boundary (reference solvers.py:17-26)
    if md.outflow_on == False:  # noqa: E712  (kept as in the reference: works for numpy bools too)
        bcs = []
    else:
        facets_outflow = locate_entities_boundary(md.domain, md.domain.topology.dim - 1, md.OutflowBoundary)
        dofs_outflow = locate_dofs_topological(md.V, md.domain.topology.dim - 1, facets_outflow)
        bc_outflow = dirichletbc(float(md.N_bdry), dofs_outflow, md.V)
        bcs = [bc_outflow]
    return bcs


_comm_ready = False


def _local_device(md):
    """The GPU of this process, decided ONCE and used for both the NCCL communicator and the model:
    LOCAL_RANK (torchrun), else OMPI_COMM_WORLD_LOCAL_RANK (mpirun, as the reference is launched),
    else rank modulo the number of visible devices; a single process keeps the current device (-1)."""
    if md.size == 1:
        return -1
    for var in ("LOCAL_RANK", "OMPI_COMM_WORLD_LOCAL_RANK", "SLURM_LOCALID"):
        if os.environ.get(var, "") != "":
            return int(os.environ[var])
    return md.rank % max(capi.device_count(), 1)


def _ensure_device_comm(md):
    """One NCCL communicator per process group, created once (replaces MPI.COMM_WORLD inside
    DOLFINx/PETSc).  The 128-byte id is broadcast with the host communicator."""
    global _comm_ready
    if md.size == 1 or _comm_ready:
        return
    uid = capi.comm_unique_id() if md.rank == 0 else None
    uid = md.comm.bcast(uid, root=0)
    capi.comm_init(uid, md.rank, md.size, _local_device(md))
    _comm_ready = True


class B200NewtonSolver:
    """What ``NewtonSolver(md.comm, NonlinearProblem(F, N, bcs))`` is in the reference
    (solvers.py:51-52): ``solve(N)`` runs the Newton iteration for the weak form of
    solvers.py:35-45 with N_n, b, q, melt_n lagged.  The fields passed in are uploaded once;
    afterwards they live on the device (``pull`` copies them back into the host Functions)."""

    # DOLFINx NewtonSolver attribute names
    rtol = 1e-9
    atol = 1e-10
    max_it = 50
    convergence_criterion = "residual"
    relaxation_parameter = 1.0

    def __init__(self, md, N, N_n, b, q, melt_n, storage, dt, bcs):
        _ensure_device_comm(md)
        self.md, self.dt = md, dt
        self.N, self.N_n, self.b, self.q, self.melt_n = N, N_n, b, q, melt_n
        opts = dict(b_min=float(md.b_min))
        opts.update(getattr(md, "solver_options", {}) or {})
        device = _local_device(md)
        self.model = capi.Model(md.domain.geometry.x[:, :2], md.domain.cells,
                                params=capi.params_from_module(params), device=device, **opts)
        m = self.model
        for name, f in (("z_b", md.z_b), ("z_s", md.z_s), ("G", md.G), ("inputs", md.inputs), ("storage", storage),
                        ("b", b), ("N", N), ("N_n", N_n), ("melt_n", melt_n)):
            m.set_field(name, f.x.array)
        m.set_flux(q.x.array)
        if bcs:
            m.set_dirichlet(np.concatenate([bc.dofs for bc in bcs]), bcs[0].value)
        self.sync_host = True       # copy N back into the Function after every solve

    def _push_newton_options(self):
        o = self.model.options
        want = (self.rtol, self.atol, self.max_it, float(self.relaxation_parameter))
        if (o.newton_rtol, o.newton_atol, o.newton_max_it, o.newton_relaxation) != want:
            self.model.set_options(newton_rtol=self.rtol, newton_atol=self.atol, newton_max_it=self.max_it,
                                   newton_relaxation=float(self.relaxation_parameter))

    def solve(self, N):
        """niter, converged = solver.solve(N)   (reference solvers.py:179).  Raises RuntimeError
        when Newton does not converge, like DOLFINx with error_on_nonconvergence."""
        self._push_newton_options()
        try:
            niter, converged = self.model.newton_solve(float(self.dt.value))
        except capi.ShaktiError as e:
            if e.code in (capi.ERR_NOT_CONVERGED, capi.ERR_LINEAR):
                raise RuntimeError(f"Newton solver did not converge: {e}") from e
            raise
        if self.sync_host:
            self.model.get_field("N", out=N.x.array)
        return niter, converged

    # the three Function.interpolate(Expression) calls of solvers.py:186-197, on the device
    def update_q(self):
        self.model.update_q()

    def update_melt(self):
        self.model.update_melt()

    def update_b(self):
        self.model.update_b(float(self.dt.value))

    def copy_N_to_N_n(self):
        self.model.copy_N_to_N_n()

    def pull(self, *names):
        """Copy device state back into the host Functions (all of it by default)."""
        names = names or ("N", "N_n", "b", "q", "melt_n")
        for k in names:
            if k == "q":
                self.q.x.array[:] = self.model.get_flux().reshape(-1)
            else:
                self.model.get_field(k, out=getattr(self, k).x.array)

    def set_inputs(self, values):
        """Replace the water-input field md.inputs on the device (time-dependent forcing, an
        extension: the reference's inputs are static, model_setup.py:47)."""
        self.model.set_field("inputs", values)

    STATE = ("N", "N_n", "b", "melt_n")

    def checkpoint(self, path, step):
        """Write the full device state (extension: the reference can only be restarted from scratch).
        On several GPUs every rank contributes its owned entries and rank 0 writes the one file, so a run
        can be resumed on any number of GPUs."""
        m = self.model
        names = list(self.STATE) + ["qx", "qy"]
        full = _sum_over_ranks(self.md, [m.get_field(k) for k in names])
        if self.md.rank == 0:
            d = dict(zip(names, full))
            q = np.stack([d.pop("qx"), d.pop("qy")], axis=1)
            np.savez(path, step=step, q=q, **d)
        self.md.comm.barrier()

    def restore(self, path):
        """Load a state written by ``checkpoint``; returns the index of the last completed step."""
        d = np.load(path)
        for k in self.STATE:
            self.model.set_field(k, d[k])
        self.model.set_flux(d["q"])
        return int(d["step"])

    def fields_for_output(self):
        """b, N, qx, qy in the caller's vertex numbering; on several GPUs every rank returns
        its owned entries and zeros elsewhere (summed by the caller)."""
        m = self.model
        return m.get_field("b"), m.get_field("N"), m.get_field("qx"), m.get_field("qy")


class _AsyncSaver:
    """The save path of reference solvers.py:199-225 without stalling the time loop: every rank
    snapshots its OWNED slice of b, N, qx, qy on the device and copies it into one of two pinned host
    buffer sets on a side stream while the next steps run (shakti_save_outputs_async); the rows reach the
    (nti, nd) arrays on rank 0 when the following save -- or a checkpoint, or the end of the run -- needs
    the buffers back."""

    def __init__(self, md, model):
        self.md, self.model = md, model
        self.owned = model.owned()                       # caller ids of this rank's dofs, device order
        self.all_owned = md.comm.gather(self.owned, root=0)
        self.sets = [[capi.PinnedArray(self.owned.size) for _ in range(4)] for _ in range(2)]
        self.pending = None                              # (row j, buffer set)
        self.k = 0

    def enqueue(self, j):
        bufs = self.sets[self.k]
        self.model.save_outputs_async(*[b.array for b in bufs], owned_only=True)
        self.pending = (j, self.k)
        self.k ^= 1

    def flush(self, arrays):
        """Wait for the pending copies and place them in row j of the four (nti, nd) arrays (rank 0)."""
        if self.pending is None:
            return
        j, k = self.pending
        self.pending = None
        self.model.wait_outputs()
        mine = [b.array for b in self.sets[k]]
        if self.md.size == 1:
            parts = [mine]
        else:
            parts = self.md.comm.gather([a.copy() for a in mine], root=0)
        if self.md.rank == 0:
            for ids, part in zip(self.all_owned, parts):
                for arr, vals in zip(arrays, part):
                    arr[j, ids] = vals


def pde_solver(md, N, N_n, b, q, melt_n, storage, dt):
    # solver for the effective pressure N (reference solvers.py:28-54)
    bcs = get_bcs(md)

    # initial guess for the Newton solver, set ONCE (reference solvers.py:48)
    N.interpolate(N_n)

    return B200NewtonSolver(md, N, N_n, b, q, melt_n, storage, dt, bcs)


def _sum_over_ranks(md, arrays):
    """Every rank holds zeros outside its owned dofs: the global field is the sum."""
    if md.size == 1:
        return arrays
    parts = md.comm.gather(arrays, root=0)
    if md.rank != 0:
        return None
    return [np.sum([p[k] for p in parts], axis=0) for k in range(len(arrays))]


def solve(md):
    # Solve the hydrology problem described by md (see setups/ for examples).
    # Results go to md.results_name:  b, qx, qy, N as (n_saved, n_dofs) arrays, t, nodes_x, nodes_y
    error_code = 0

    nt = np.size(md.timesteps)
    dt_ = 0.1 * np.abs(md.timesteps[1] - md.timesteps[0])
    dt = Constant(md.domain, dt_)

    # node coordinates in the order the solution arrays are saved
    nodes_x = md.comm.gather(md.x[md.mask], root=0)
    nodes_y = md.comm.gather(md.y[md.mask], root=0)

    md.comm.barrier()
    if md.rank == 0:
        try:
            os.makedirs(md.results_name, exist_ok=bool(getattr(md, "resume", False)))
        except FileExistsError:
            print(f"Error: Directory '{md.results_name}' already exists.\n"
                  "Choose another name in setup file or delete this directory.")
            error_code = 1

    md.comm.barrier()
    error_code = md.comm.bcast(error_code, root=0)

    if error_code == 1:
        sys.exit(1)

    if md.rank == 0:
        parent_dir = str((Path(__file__).resolve()).parent.parent)
        nodes_x = nodes_x[0]       # every process holds the whole mesh: no concatenation needed
        nodes_y = nodes_y[0]
        nti = int(nt / md.nt_save)
        t_i = np.linspace(0, md.timesteps.max(), nti)
        nd = md.V.dofmap.index_map.size_global

        b_arr = np.zeros((nti, nd))
        N_arr = np.zeros((nti, nd))
        qx_arr = np.zeros((nti, nd))
        qy_arr = np.zeros((nti, nd))

        np.save(md.results_name + '/t.npy', t_i)
        np.save(md.results_name + '/nodes_x.npy', nodes_x)
        np.save(md.results_name + '/nodes_y.npy', nodes_y)

        # keep a copy of the setup file next to the results
        src = parent_dir + '/setups/{}.py'.format(md.setup_name)
        if os.path.exists(src):
            shutil.copy(src, md.results_name + '/{}.py'.format(md.setup_name))
        j = 0

    # solution functions and initial conditions
    N = Function(md.V)
    q = Function(md.V_flux)
    b = Function(md.V)
    N_n = Function(md.V)

    b.interpolate(md.b_init)
    N_n.interpolate(md.N_init)
    q.sub(0).interpolate(md.q_init.sub(0))
    q.sub(1).interpolate(md.q_init.sub(1))

    if md.storage_on == False:  # noqa: E712
        storage = Function(md.V)        # zero: storage term switched off
    else:
        storage = md.lake_bdry

    melt_n = Function(md.V)             # melt rate at the previous step (Warburton et al. 2024 term)

    solver = pde_solver(md, N, N_n, b, q, melt_n, storage, dt)
    solver.sync_host = False            # state stays on the device between saves
    md.solver = solver
    saver = _AsyncSaver(md, solver.model)
    out_arrays = (b_arr, N_arr, qx_arr, qy_arr) if md.rank == 0 else None
    if md.rank != 0:
        j = 0

    # extensions (off unless the setup sets them): md.inputs_of_t(t) -> nodal array for time-dependent
    # forcing, md.resume = True to continue from <results>/checkpoint.npz written every nt_check saves
    inputs_of_t = getattr(md, "inputs_of_t", None)
    first = 0
    ckpt = os.path.join(md.results_name, "checkpoint.npz")
    if getattr(md, "resume", False) and os.path.exists(ckpt):
        first = solver.restore(ckpt) + 1
        if md.rank == 0:
            for name, arr in (("b", b_arr), ("N", N_arr), ("qx", qx_arr), ("qy", qy_arr)):
                old = os.path.join(md.results_name, name + ".npy")
                if os.path.exists(old):
                    prev = np.load(old)
                    arr[:min(arr.shape[0], prev.shape[0])] = prev[:arr.shape[0]]
        j = len(range(0, first, md.nt_save))

    # extension (off unless md.diagnostics_on): one water-budget record per time step (capi.DIAGNOSTICS), recorded on
    # the device and written by rank 0 to <results>/diagnostics.npz (t and one array per column) at every checkpoint
    # save and at the end; a resumed run keeps the rows of the steps before `first` from the existing file
    diag = None
    if getattr(md, "diagnostics_on", False):
        solver.model.record_diagnostics(max(nt - first, 1))
        diag_file = os.path.join(md.results_name, "diagnostics.npz")
        diag = dict(t=np.zeros(0), rows=np.zeros((0, len(capi.DIAGNOSTICS))), read=0)
        if first > 0 and md.rank == 0 and os.path.exists(diag_file):
            prev = np.load(diag_file)
            diag["t"] = prev["t"][:first]
            diag["rows"] = np.stack([prev[k] for k in capi.DIAGNOSTICS], axis=1)[:first]

    def save_diagnostics():
        rows = solver.model.read_diagnostics()      # every rank: the records are global and each rank empties its buffer
        i0 = first + diag["read"]
        diag["read"] += rows.shape[0]
        if md.rank == 0:
            diag["t"] = np.concatenate([diag["t"], md.timesteps[i0:i0 + rows.shape[0]]])
            diag["rows"] = np.concatenate([diag["rows"], rows])
            np.savez(diag_file, t=diag["t"], **dict(zip(capi.DIAGNOSTICS, diag["rows"].T)))

    for i in range(first, nt):

        if md.rank == 0 and (i + 1) % 10 == 0:
            print(f"Time step {i+1} of {nt} completed ({(i+1)/nt*100:.1f}%)", end='\r')
            sys.stdout.flush()

        if i > 0:
            dt_ = np.abs(md.timesteps[i] - md.timesteps[i - 1])
            dt.value = dt_

        if inputs_of_t is not None:
            solver.set_inputs(inputs_of_t(md.timesteps[i]))

        # effective pressure
        niter, converged = solver.solve(N)
        assert (converged)

        # water flux, melt rate, gap height (with lower bound b_min), on the device
        solver.update_q()
        solver.update_melt()
        solver.update_b()

        if i % md.nt_save == 0:
            # the previous save's rows come home now (their copies overlapped the steps in between),
            # then this step's fields are snapshotted on the device and start their way to the host
            saver.flush(out_arrays)
            saver.enqueue(j)

            if i % md.nt_check == 0:
                # checkpoint: lets plots be made while the run is in progress (needs this row now)
                saver.flush(out_arrays)
                if md.rank == 0:
                    np.save(md.results_name + '/b.npy', b_arr)
                    np.save(md.results_name + '/N.npy', N_arr)
                    np.save(md.results_name + '/qx.npy', qx_arr)
                    np.save(md.results_name + '/qy.npy', qy_arr)
                if diag is not None:
                    save_diagnostics()

            j += 1

            if i % md.nt_check == 0 and getattr(md, "resume", False):
                solver.copy_N_to_N_n()          # the checkpoint holds the state the next step starts from
                solver.checkpoint(ckpt, i)

        # previous-step solution
        solver.copy_N_to_N_n()

    saver.flush(out_arrays)
    if md.rank == 0:
        np.save(md.results_name + '/b.npy', b_arr)
        np.save(md.results_name + '/N.npy', N_arr)
        np.save(md.results_name + '/qx.npy', qx_arr)
        np.save(md.results_name + '/qy.npy', qy_arr)
    if diag is not None:
        save_diagnostics()

    solver.pull()
    md.final = dict(N=N, N_n=N_n, b=b, q=q, melt_n=melt_n)
    return
