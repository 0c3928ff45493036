"""ctypes binding of ``include/shakti_b200.h`` (the C ABI of the CUDA library).

Thin by design: numpy arrays / raw pointers in, numpy arrays out, every non-zero return code
re-raised as ``ShaktiError`` with the library's message.  There is no CPU fallback: if the
shared library is missing, or no sm_100 GPU is visible, the calls fail loudly.
"""
import ctypes as C
import os
from pathlib import Path

import numpy as np

_ROOT = Path(__file__).resolve().parent.parent
LIB_PATH = _ROOT / "lib" / "libshakti_b200.so"

FIELDS = dict(z_b=0, z_s=1, G=2, inputs=3, storage=4, b=5, N=6, N_n=7, qx=8, qy=9, melt_n=10, residual=11)
KSP = dict(gmres=0, bicgstab=1)
PC = dict(jacobi=0, amg=1, none=2)
NEWTON_R0 = dict(dolfinx=0, initial_residual=1)
HOST_ARRAYS = dict(l2g=0, cells=1, cell_l2g=2, rowptr=3, col=4, slice_ptr=5, sell_col=6, slot=7, diag_pos=8,
                   win=9, win_cell=10, nbr_rank=11, nbr_send_ptr=12, nbr_send_idx=13, nbr_recv=14,
                   ab_info=15, ab_eptr=16, ab_elems=17, ab_lv=18, ab_hptr=19, ab_halo=20, ab_incptr=21, ab_inc=22, ab_src=23,
                   cell_counted=24)
# columns of a water-budget record (enum shakti_diag)
DIAGNOSTICS = ("dt", "newton_its", "residual", "area", "water_volume", "input", "melt", "closure", "storage", "outflow",
               "imbalance", "N_mean", "N_min", "N_max", "b_max")

ERR_NOT_CONVERGED = -4
ERR_LINEAR = -5


class ShaktiError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"[shakti_b200 {code}] {msg}")
        self.code = code


class Params(C.Structure):
    """source/params.py:4-11"""
    _fields_ = [(k, C.c_double) for k in ("g", "rho_i", "rho_w", "nu", "Lh", "omega", "n", "A")]


class Options(C.Structure):
    _fields_ = [
        ("newton_rtol", C.c_double), ("newton_atol", C.c_double),
        ("newton_max_it", C.c_int32), ("newton_r0", C.c_int32),
        ("linear_solver", C.c_int32), ("precond", C.c_int32),
        ("linear_rtol", C.c_double), ("linear_atol", C.c_double),
        ("linear_max_it", C.c_int32), ("gmres_restart", C.c_int32),
        ("amg_refresh_every", C.c_int32), ("amg_max_levels", C.c_int32),
        ("amg_coarse_size", C.c_int32), ("amg_presmooth", C.c_int32), ("amg_postsmooth", C.c_int32),
        ("amg_smoother_omega", C.c_double), ("amg_prolong_omega", C.c_double),
        ("amg_strength_theta", C.c_double), ("amg_cheby_ratio", C.c_double),
        ("amg_smoother", C.c_int32), ("amg_fp32_cycle", C.c_int32),
        ("amg_cuda_graph", C.c_int32), ("amg_smoother_halo", C.c_int32),
        ("b_min", C.c_double), ("assembly_kernel", C.c_int32), ("reorder", C.c_int32),
        ("linear_forcing", C.c_double), ("amg_replicate_below", C.c_int32),
        ("newton_relaxation", C.c_double), ("newton_line_search", C.c_int32),
    ]


class Stats(C.Structure):
    _fields_ = [(k, C.c_int64) for k in (
        "n_vert", "n_cell", "nnz", "n_owned", "n_local", "n_cell_local", "nnz_local", "steps", "newton_its",
        "linear_its", "kernel_launches", "amg_levels", "amg_refreshes")] + [
        (k, C.c_double) for k in ("amg_operator_complexity", "last_residual", "last_residual0", "last_linear_relres")] + [
        ("newton_backtracks", C.c_int64)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


_lib = None


def load():
    """Load the shared library (raises if it has not been built)."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise ShaktiError(-2, f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                              "or `make -C shakti-fenics_b200/csrc` (there is no CPU fallback)")
    lib = C.CDLL(str(LIB_PATH), mode=os.RTLD_GLOBAL if hasattr(os, "RTLD_GLOBAL") else C.DEFAULT_MODE)
    lib.shakti_last_error.restype = C.c_char_p
    lib.shakti_version.restype = C.c_char_p
    _lib = lib
    return lib


def _check(rc):
    if rc != 0:
        raise ShaktiError(rc, load().shakti_last_error().decode())


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def device_count():
    n = C.c_int(0)
    _check(load().shakti_device_count(C.byref(n)))
    return n.value


def default_params():
    p = Params()
    _check(load().shakti_default_params(C.byref(p)))
    return p


def params_from_module(mod):
    """Build the constant struct from a ``params`` module (reference source/params.py)."""
    p = Params()
    for k, _ in Params._fields_:
        setattr(p, k, float(getattr(mod, k)))
    return p


def default_options(**kw):
    o = Options()
    _check(load().shakti_default_options(C.byref(o)))
    _apply_options(o, kw)
    return o


def _apply_options(o, kw):
    names = {k for k, _ in Options._fields_}
    for k, v in kw.items():
        if k not in names:
            raise KeyError(f"unknown option {k!r}")
        if k == "linear_solver" and isinstance(v, str):
            v = KSP[v]
        if k == "precond" and isinstance(v, str):
            v = PC[v]
        if k == "newton_r0" and isinstance(v, str):
            v = NEWTON_R0[v]
        if k == "amg_smoother" and isinstance(v, str):
            v = dict(jacobi=0, chebyshev=1)[v]
        setattr(o, k, v)


# ---------------------------------------------------------------------------- host helpers
def host_csr_pattern(n_vert, cells):
    lib = load()
    cells = _i32(cells)
    nnz = C.c_int64(0)
    _check(lib.shakti_host_csr_pattern(C.c_int64(n_vert), C.c_int64(cells.shape[0]), _p(cells), None, None, C.byref(nnz)))
    rowptr = np.empty(n_vert + 1, dtype=np.int32)
    col = np.empty(nnz.value, dtype=np.int32)
    _check(lib.shakti_host_csr_pattern(C.c_int64(n_vert), C.c_int64(cells.shape[0]), _p(cells), _p(rowptr), _p(col), C.byref(nnz)))
    return rowptr, col


def host_locate_dirichlet(n_vert, cells, marker):
    lib = load()
    cells = _i32(cells)
    marker = np.ascontiguousarray(marker, dtype=np.uint8)
    n = C.c_int64(0)
    out = np.empty(n_vert, dtype=np.int32)
    _check(lib.shakti_host_locate_dirichlet(C.c_int64(n_vert), C.c_int64(cells.shape[0]), _p(cells), _p(marker),
                                            _p(out), C.c_int64(n_vert), C.byref(n)))
    return out[: n.value].copy()


def host_amg_aggregate(A_csr, theta=0.08, exclude=None):
    """Aggregates of a scipy CSR matrix as the AMG set-up forms them -> (agg ids, count)."""
    lib = load()
    n = A_csr.shape[0]
    rp, col, val = _i32(A_csr.indptr), _i32(A_csr.indices), _f64(A_csr.data)
    agg = np.empty(n, dtype=np.int32)
    na = C.c_int32(0)
    ex = None if exclude is None else np.ascontiguousarray(exclude, dtype=np.uint8)
    _check(lib.shakti_host_amg_aggregate(C.c_int32(n), _p(rp), _p(col), _p(val), C.c_double(theta),
                                         _p(ex) if ex is not None else None, _p(agg), C.byref(na)))
    return agg, na.value


class HostMesh:
    """The rank-local mesh the device code works on (host-only; no GPU needed)."""

    def __init__(self, xy, cells, rank=0, nranks=1, reorder=1):
        lib = load()
        xy, cells = _f64(xy), _i32(cells)
        self._h = C.c_void_p()
        _check(lib.shakti_host_mesh_create(C.c_int64(xy.shape[0]), C.c_int64(cells.shape[0]), _p(xy), _p(cells),
                                           C.c_int(rank), C.c_int(nranks), C.c_int(reorder), C.byref(self._h)))
        info = (C.c_int64 * 6)()
        _check(lib.shakti_host_mesh_info(self._h, info))
        self.n_owned, self.n_local, self.n_cell, self.nnz, self.padded, self.n_nbrs = [int(v) for v in info]

    def array(self, name):
        lib = load()
        n = C.c_int64(0)
        _check(lib.shakti_host_mesh_array(self._h, C.c_int(HOST_ARRAYS[name]), None, C.byref(n)))
        out = np.empty(n.value, dtype=np.int32)
        _check(lib.shakti_host_mesh_array(self._h, C.c_int(HOST_ARRAYS[name]), _p(out), C.byref(n)))
        return out

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.shakti_host_mesh_destroy(self._h)
            self._h = None


def interp_grid(px, py, xg, yg, f_yx):
    """Bilinear interpolation / linear extrapolation of f_yx[iy, ix] at points (px, py) on the GPU."""
    px, py, xg, yg, f = _f64(px), _f64(py), _f64(xg), _f64(yg), _f64(f_yx)
    assert f.shape == (yg.size, xg.size)
    out = np.empty(px.size)
    _check(load().shakti_interp_grid(C.c_int64(px.size), _p(px), _p(py), C.c_int32(xg.size), C.c_int32(yg.size), _p(xg), _p(yg),
                                     _p(f), _p(out)))
    return out


def points_in_polygon(px, py, poly):
    """1.0 / 0.0 per point: inside the closed polygon poly (m, 2) by the even-odd rule, on the GPU."""
    px, py, poly = _f64(px), _f64(py), _f64(poly)
    out = np.empty(px.size)
    _check(load().shakti_points_in_polygon(C.c_int64(px.size), _p(px), _p(py), C.c_int32(poly.shape[0]), _p(poly), _p(out)))
    return out


class PinnedArray:
    """A float64 numpy array over page-locked host memory (cudaMallocHost), freed with the object."""

    def __init__(self, n):
        self._lib = load()
        self._ptr = C.c_void_p()
        _check(self._lib.shakti_alloc_pinned(C.c_int64(8 * max(int(n), 1)), C.byref(self._ptr)))
        buf = (C.c_double * max(int(n), 1)).from_address(self._ptr.value)
        self.array = np.frombuffer(buf, dtype=np.float64)[: int(n)]

    def __del__(self):
        try:
            if getattr(self, "_ptr", None) and self._ptr.value:
                self.array = None
                self._lib.shakti_free_pinned(self._ptr)
                self._ptr = C.c_void_p()
        except Exception:
            pass


# ---------------------------------------------------------------------------- multi-GPU
def comm_unique_id():
    buf = (C.c_uint8 * 128)()
    _check(load().shakti_comm_unique_id(buf))
    return bytes(buf)


def comm_init(uid, rank, nranks, device=-1):
    buf = (C.c_uint8 * 128).from_buffer_copy(uid)
    _check(load().shakti_comm_init(buf, C.c_int(rank), C.c_int(nranks), C.c_int(device)))


def comm_finalize():
    _check(load().shakti_comm_finalize())


# ---------------------------------------------------------------------------- the model
class Model:
    """Owner of one ``shakti_model`` handle.  Array arguments are numpy (host) arrays in the
    caller's vertex numbering unless a method says ``ptr`` (raw device/pinned pointer)."""

    def __init__(self, xy, cells, params=None, options=None, device=-1, **opt_kw):
        self.lib = load()
        xy, cells = _f64(xy), _i32(cells)
        assert xy.ndim == 2 and xy.shape[1] == 2 and cells.ndim == 2 and cells.shape[1] == 3
        self.n_vert, self.n_cell = int(xy.shape[0]), int(cells.shape[0])
        self.params = params or default_params()
        self.options = options or default_options()
        _apply_options(self.options, opt_kw)
        self._h = C.c_void_p()
        _check(self.lib.shakti_create(C.c_int64(self.n_vert), C.c_int64(self.n_cell), _p(xy), _p(cells),
                                      C.byref(self.params), C.byref(self.options), C.c_int(device), C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None):
            self.lib.shakti_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- options / stats
    def set_options(self, **kw):
        _apply_options(self.options, kw)
        _check(self.lib.shakti_set_options(self._h, C.byref(self.options)))

    def stats(self):
        st = Stats()
        _check(self.lib.shakti_get_stats(self._h, C.byref(st)))
        return st.as_dict()

    # ---- data in/out
    def set_field(self, name, values):
        v = _f64(values)
        if v.ndim == 0:
            v = np.full(self.n_vert, float(v))
        assert v.shape == (self.n_vert,), (name, v.shape)
        _check(self.lib.shakti_set_field(self._h, C.c_int(FIELDS[name]), _p(v), C.c_int(0)))

    def get_field(self, name, out=None):
        out = np.empty(self.n_vert) if out is None else out
        _check(self.lib.shakti_get_field(self._h, C.c_int(FIELDS[name]), _p(out), C.c_int(0)))
        return out

    def set_field_ptr(self, name, ptr, is_device):
        _check(self.lib.shakti_set_field(self._h, C.c_int(FIELDS[name]), C.c_void_p(ptr), C.c_int(is_device)))

    def get_field_ptr(self, name, ptr, is_device):
        _check(self.lib.shakti_get_field(self._h, C.c_int(FIELDS[name]), C.c_void_p(ptr), C.c_int(is_device)))

    def set_flux(self, q):
        q = _f64(q).reshape(-1)
        assert q.size == 2 * self.n_vert
        _check(self.lib.shakti_set_flux(self._h, _p(q), C.c_int(0)))

    def get_flux(self):
        q = np.empty(2 * self.n_vert)
        _check(self.lib.shakti_get_flux(self._h, _p(q), C.c_int(0)))
        return q.reshape(-1, 2)

    def set_dirichlet(self, dofs, value):
        d = _i32(dofs)
        _check(self.lib.shakti_set_dirichlet(self._h, _p(d), C.c_int64(d.size), C.c_double(value)))

    def locate_dirichlet(self, marker):
        marker = np.ascontiguousarray(marker, dtype=np.uint8)
        out = np.empty(self.n_vert, dtype=np.int32)
        n = C.c_int64(0)
        _check(self.lib.shakti_locate_dirichlet(self._h, _p(marker), _p(out), C.c_int64(self.n_vert), C.byref(n)))
        return out[: n.value].copy()

    def interp_grid_to_field(self, name, xg, yg, f_yx):
        xg, yg, f = _f64(xg), _f64(yg), _f64(f_yx)
        assert f.shape == (yg.size, xg.size)
        _check(self.lib.shakti_interp_grid_to_field(self._h, C.c_int(FIELDS[name]), C.c_int32(xg.size), C.c_int32(yg.size),
                                                    _p(xg), _p(yg), _p(f)))

    def polygon_to_field(self, name, poly):
        poly = _f64(poly)
        _check(self.lib.shakti_polygon_to_field(self._h, C.c_int(FIELDS[name]), C.c_int32(poly.shape[0]), _p(poly)))

    def set_quadrature(self, pts, wts):
        pts, wts = _f64(pts), _f64(wts)
        _check(self.lib.shakti_set_quadrature(self._h, C.c_int32(wts.size), _p(pts), _p(wts)))

    # ---- parity hooks
    def csr(self):
        nnz = C.c_int64(0)
        _check(self.lib.shakti_get_csr(self._h, None, None, C.byref(nnz)))
        rowptr = np.empty(self.n_vert + 1, dtype=np.int32)
        col = np.empty(nnz.value, dtype=np.int32)
        _check(self.lib.shakti_get_csr(self._h, _p(rowptr), _p(col), C.byref(nnz)))
        return rowptr, col

    def kbar(self):
        out = np.empty(self.n_cell)
        _check(self.lib.shakti_kbar(self._h, _p(out)))
        return out

    def assemble(self, dt, want_J=True):
        F = np.empty(self.n_vert)
        if want_J:
            nnz = C.c_int64(0)
            _check(self.lib.shakti_get_csr(self._h, None, None, C.byref(nnz)))
            J = np.empty(nnz.value)
            _check(self.lib.shakti_assemble(self._h, C.c_double(dt), _p(F), _p(J)))
            return F, J
        _check(self.lib.shakti_assemble(self._h, C.c_double(dt), _p(F), None))
        return F, None

    def spmv(self, x):
        x = _f64(x)
        y = np.empty(self.n_vert)
        _check(self.lib.shakti_spmv(self._h, _p(x), _p(y)))
        return y

    def linear_solve(self, rhs):
        rhs = _f64(rhs)
        dx = np.empty(self.n_vert)
        it, rr = C.c_int32(0), C.c_double(0)
        _check(self.lib.shakti_linear_solve(self._h, _p(rhs), _p(dx), C.byref(it), C.byref(rr)))
        return dx, it.value, rr.value

    def winning_cells(self):
        out = np.empty(self.n_vert, dtype=np.int32)
        _check(self.lib.shakti_get_winning_cells(self._h, _p(out)))
        return out

    def owned(self):
        n = C.c_int64(0)
        _check(self.lib.shakti_get_owned(self._h, None, C.byref(n)))
        ids = np.empty(n.value, dtype=np.int32)
        _check(self.lib.shakti_get_owned(self._h, _p(ids), C.byref(n)))
        return ids

    # ---- hot path
    def start(self):
        _check(self.lib.shakti_start(self._h))

    def newton_solve(self, dt):
        it, cv = C.c_int32(0), C.c_int32(0)
        _check(self.lib.shakti_newton_solve(self._h, C.c_double(dt), C.byref(it), C.byref(cv)))
        return it.value, bool(cv.value)

    def update_q(self):
        _check(self.lib.shakti_update_q(self._h))

    def update_melt(self):
        _check(self.lib.shakti_update_melt(self._h))

    def update_q_melt(self):
        _check(self.lib.shakti_update_q_melt(self._h))

    def update_b(self, dt):
        _check(self.lib.shakti_update_b(self._h, C.c_double(dt)))

    def copy_N_to_N_n(self):
        _check(self.lib.shakti_copy_N_to_N_n(self._h))

    def snapshot(self):
        _check(self.lib.shakti_snapshot(self._h))

    def rollback(self):
        _check(self.lib.shakti_rollback(self._h))

    def step(self, dt):
        it, cv = C.c_int32(0), C.c_int32(0)
        _check(self.lib.shakti_step(self._h, C.c_double(dt), C.byref(it), C.byref(cv)))
        return it.value, bool(cv.value)

    def run(self, dts):
        dts = _f64(dts)
        its = np.zeros(dts.size, dtype=np.int32)
        _check(self.lib.shakti_run(self._h, _p(dts), C.c_int64(dts.size), _p(its)))
        return its

    def run_timed(self, dts):
        """run() bracketed by CUDA events on the library stream -> (niter per step, milliseconds)."""
        dts = _f64(dts)
        its = np.zeros(dts.size, dtype=np.int32)
        ms = C.c_double(0)
        _check(self.lib.shakti_run_timed(self._h, _p(dts), C.c_int64(dts.size), _p(its), C.byref(ms)))
        return its, ms.value

    def step_host(self, dt, inputs_ptr=None, b_ptr=None, N_ptr=None, qx_ptr=None, qy_ptr=None):
        """shakti_step_host with raw host pointers (e.g. pinned torch tensors' data_ptr())."""
        it, cv = C.c_int32(0), C.c_int32(0)
        vp = lambda p: C.c_void_p(p) if p else None
        _check(self.lib.shakti_step_host(self._h, C.c_double(dt), vp(inputs_ptr), vp(b_ptr), vp(N_ptr), vp(qx_ptr),
                                         vp(qy_ptr), C.byref(it), C.byref(cv)))
        return it.value, bool(cv.value)

    def step_host_async(self, dt, inputs_ptr=None, b_ptr=None, N_ptr=None, qx_ptr=None, qy_ptr=None, owned_only=False):
        """shakti_step_host_async: the D2H copies are only enqueued; call wait_outputs() before reading."""
        it, cv = C.c_int32(0), C.c_int32(0)
        vp = lambda p: C.c_void_p(p) if p else None
        _check(self.lib.shakti_step_host_async(self._h, C.c_double(dt), vp(inputs_ptr), vp(b_ptr), vp(N_ptr), vp(qx_ptr),
                                               vp(qy_ptr), C.c_int(1 if owned_only else 0), C.byref(it), C.byref(cv)))
        return it.value, bool(cv.value)

    def wait_outputs(self):
        _check(self.lib.shakti_wait_outputs(self._h))

    def save_outputs_async(self, b, N, qx, qy, owned_only=False):
        """Enqueue snapshots of b, N, qx, qy into the given (pinned) numpy arrays; valid after wait_outputs()."""
        _check(self.lib.shakti_save_outputs_async(self._h, _p(b), _p(N), _p(qx), _p(qy), C.c_int(1 if owned_only else 0)))

    # ---- water-budget diagnostics (columns: DIAGNOSTICS)
    def diagnostics(self, dt):
        """One record of the current state -> dict (columns 0-2: dt, 0, ||F|| of the current state)."""
        out = np.empty(len(DIAGNOSTICS))
        _check(self.lib.shakti_diagnostics(self._h, C.c_double(dt), _p(out)))
        return dict(zip(DIAGNOSTICS, out.tolist()))

    def record_diagnostics(self, capacity):
        """capacity > 0: every converged Newton solve appends one record on the device; 0: off."""
        _check(self.lib.shakti_record_diagnostics(self._h, C.c_int64(int(capacity))))

    def read_diagnostics(self):
        """The recorded rows as an (n, len(DIAGNOSTICS)) array; empties the buffer."""
        n = C.c_int64(0)
        _check(self.lib.shakti_read_diagnostics(self._h, None, C.c_int64(0), C.byref(n)))
        rows = np.empty((n.value, len(DIAGNOSTICS)))
        _check(self.lib.shakti_read_diagnostics(self._h, _p(rows), C.c_int64(n.value), C.byref(n)))
        return rows[: n.value]

    # ---- moulins (point water inputs with hydrographs; see shakti_set_moulins in the header)
    def set_moulins(self, vertex, times, discharges, period=0.0, knot_ptr=None):
        """Moulin k at caller vertex ``vertex[k]`` with hydrograph knots ``(times[k][j], discharges[k][j])`` [s, m^3/s].
        ``times`` / ``discharges`` are ragged lists (one sequence per moulin), or flat arrays with ``knot_ptr`` (CSR,
        len(vertex) + 1 entries).  ``period`` > 0 wraps t into [t_0, t_0 + period) of each hydrograph.  An empty
        ``vertex`` removes every moulin."""
        v = _i32(vertex).reshape(-1)
        if knot_ptr is None:
            if len(times) != v.size or len(discharges) != v.size:
                raise ValueError("one hydrograph (times, discharges) per moulin")
            lens = [np.size(t) for t in times]
            if any(np.size(q) != n for q, n in zip(discharges, lens)):
                raise ValueError("times and discharges of a moulin differ in length")
            kp = np.zeros(v.size + 1, dtype=np.int64)
            kp[1:] = np.cumsum(lens)
            tk = _f64(np.concatenate([np.ravel(t) for t in times]) if v.size else np.zeros(0))
            qk = _f64(np.concatenate([np.ravel(q) for q in discharges]) if v.size else np.zeros(0))
        else:
            kp = np.ascontiguousarray(knot_ptr, dtype=np.int64)
            tk, qk = _f64(times).reshape(-1), _f64(discharges).reshape(-1)
            if kp.size != v.size + 1 or tk.size != qk.size or (v.size and (kp[0] != 0 or kp[-1] != tk.size)):
                raise ValueError("knot_ptr must have len(vertex) + 1 entries from 0 to the number of knots")
        _check(self.lib.shakti_set_moulins(self._h, C.c_int64(v.size), _p(v), _p(kp), _p(tk), _p(qk), C.c_double(period)))
        self.n_moulins = int(v.size)

    def set_time(self, t):
        """Model clock [s]: a solve with step dt is forced at t + dt; update_b advances the clock by dt."""
        _check(self.lib.shakti_set_time(self._h, C.c_double(t)))

    def get_time(self):
        t = C.c_double(0)
        _check(self.lib.shakti_get_time(self._h, C.byref(t)))
        return t.value

    def moulin_discharge(self, t):
        """Q_k(t) of every moulin, in the order given to set_moulins."""
        q = np.empty(getattr(self, "n_moulins", 0))
        _check(self.lib.shakti_moulin_discharge(self._h, C.c_double(t), _p(q)))
        return q

    # ---- micro-benchmarks
    KERNELS = dict(spmv=0, assemble=1, kbar=2, nodal=3, dot=4, axpy=5)

    def time_kernel(self, which, reps=20, dt=3600.0):
        ms = C.c_double(0)
        _check(self.lib.shakti_time_kernel(self._h, C.c_int(self.KERNELS[which]), C.c_int(reps), C.c_double(dt), C.byref(ms)))
        return ms.value

    def time_amg_smoother(self, level, reps=20):
        """-> dict(ms, rows, nnz, value_bytes, bytes) for one smoothing step of AMG level `level`."""
        ms, rows, nnz, vb, xb = C.c_double(0), C.c_int64(0), C.c_int64(0), C.c_int32(0), C.c_int32(0)
        _check(self.lib.shakti_time_amg_smoother(self._h, C.c_int(level), C.c_int(reps), C.byref(ms), C.byref(rows),
                                                 C.byref(nnz), C.byref(vb), C.byref(xb)))
        by = (vb.value + 4) * nnz.value + 7 * xb.value * rows.value
        return dict(ms=ms.value, rows=rows.value, nnz=nnz.value, value_bytes=vb.value, vector_bytes=xb.value, bytes=by)

    AMG_LEVEL_KERNELS = {"smoother": 0, "residual": 1, "restriction": 2, "prolongation": 3}

    def time_amg_level_kernel(self, level, which, reps=20):
        """-> dict(ms, rows, cols, nnz, max_width, value_bytes, vector_bytes, fused) for one launch of SELL kernel
        `which` (AMG_LEVEL_KERNELS) of AMG level `level`, launched as the V-cycle launches it; the shape and value
        bytes are those of the kernel's matrix (A, R or P); fused: the restriction takes the coarse level's first
        Chebyshev step too."""
        ms, info = C.c_double(0), (C.c_int64 * 7)()
        _check(self.lib.shakti_time_amg_level_kernel(self._h, C.c_int(level), C.c_int(self.AMG_LEVEL_KERNELS[which]),
                                                     C.c_int(reps), C.byref(ms), info))
        return dict(ms=ms.value, rows=info[0], cols=info[1], nnz=info[2], max_width=info[3], value_bytes=info[4],
                    vector_bytes=info[5], fused=bool(info[6]))

    def kernel_bytes(self, which):
        b = C.c_double(0)
        _check(self.lib.shakti_kernel_bytes(self._h, C.c_int(self.KERNELS[which]), C.byref(b)))
        return b.value

    # ---- AMG test hooks (one rank; internal order: owned() gives the caller id of each row)
    AMG_INFO = ("rows", "cols", "n_coarse", "A_nnz", "A_width", "P_nnz", "P_width", "R_nnz", "R_width", "last",
                "dense_coarse", "uses_half", "restrict_starts", "seams_apply", "levels", "fp32_cycle", "table_AP",
                "table_RAP")
    AMG_MATRICES = dict(A=0, P=1, R=2, valf=3, valh=4)

    def amg_refresh(self, full=True):
        """Rebuild the AMG preconditioner from the last assembled Jacobian: the whole hierarchy (full) or only the
        fine smoother, the rest lagged."""
        _check(self.lib.shakti_amg_refresh(self._h, C.c_int(1 if full else 0)))

    def amg_level_info(self, level):
        info = (C.c_int64 * len(self.AMG_INFO))()
        _check(self.lib.shakti_amg_level_info(self._h, C.c_int(level), info))
        return dict(zip(self.AMG_INFO, (int(v) for v in info)))

    def amg_matrix(self, level, which):
        """Matrix `which` (AMG_MATRICES) of AMG level `level` -> scipy CSR in internal order, values as double."""
        import scipy.sparse as sp
        k = C.c_int(self.AMG_MATRICES[which])
        nnz = C.c_int64(0)
        _check(self.lib.shakti_amg_get_matrix(self._h, C.c_int(level), k, None, None, None, C.byref(nnz)))
        info = self.amg_level_info(level)
        rows, cols = info["rows"], info["cols"]
        if which == "P":
            cols = info["n_coarse"]
        elif which == "R":
            rows = info["n_coarse"]
        rowptr = np.empty(rows + 1, dtype=np.int32)
        col = np.empty(nnz.value, dtype=np.int32)
        val = np.empty(nnz.value)
        _check(self.lib.shakti_amg_get_matrix(self._h, C.c_int(level), k, _p(rowptr), _p(col), _p(val), C.byref(nnz)))
        return sp.csr_matrix((val, col, rowptr), shape=(rows, cols))

    def amg_vectors(self, level):
        """-> dict(dinv, dinv_cycle, lmax, coef) of AMG level `level` (coef: empty without the Chebyshev smoother)."""
        n = self.amg_level_info(level)["rows"]
        dinv, dc = np.empty(n), np.empty(n)
        lmax, stride = C.c_double(0), C.c_int32(0)
        _check(self.lib.shakti_amg_get_vectors(self._h, C.c_int(level), None, None, None, None, C.byref(stride)))
        coef = np.empty(stride.value)
        _check(self.lib.shakti_amg_get_vectors(self._h, C.c_int(level), _p(dinv), _p(dc), C.byref(lmax), _p(coef),
                                               C.byref(stride)))
        return dict(dinv=dinv, dinv_cycle=dc, lmax=lmax.value, coef=coef)

    def amg_apply(self, r):
        """z = M^-1 r: one V-cycle on owned-length vectors in internal order, as a Krylov iteration applies it."""
        r = _f64(r)
        z = np.empty_like(r)
        _check(self.lib.shakti_amg_apply(self._h, _p(r), _p(z)))
        return z
