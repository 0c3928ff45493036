"""Seeded synthetic inputs for the BASELINE.json configs (SURVEY.md §8d).

Every builder returns a ``Case``: the mesh arrays, the vertex fields of ``model_setup``
(reference source/model_setup.py:44-53), the Dirichlet dofs of ``get_bcs``
(source/solvers.py:17-26) and a ``timesteps`` array (setups/setup_cooke2.py:92-95).
"""
from dataclasses import dataclass, field

import numpy as np

from . import meshgen


@dataclass
class Case:
    name: str
    xy: np.ndarray
    cells: np.ndarray
    fields: dict
    bc_dofs: np.ndarray
    N_bdry: float
    timesteps: np.ndarray
    storage_on: bool = False
    meta: dict = field(default_factory=dict)

    @property
    def n_vert(self):
        return self.xy.shape[0]

    def dts(self, n=None):
        """solvers.py:81,174-176: first step 0.1*|t1-t0|, then |t_i - t_{i-1}|."""
        t = self.timesteps
        d = np.empty(t.size)
        d[0] = 0.1 * abs(t[1] - t[0])
        d[1:] = np.abs(t[1:] - t[:-1])
        return d if n is None else d[:n]


def _left_edge_dofs(nx, ny):
    """vertices with x == x0 on the structured generator's numbering (iy*(nx+1))"""
    return (np.arange(ny + 1, dtype=np.int64) * (nx + 1)).astype(np.int32)


def _smooth_bed(x, y, lx, ly, amp, rng, modes=8):
    """Sum of `modes` cosine products.  Element-wise, so large meshes are evaluated in chunks on a few threads
    (numpy releases the GIL): the 256M cosines of the 16M-dof case were half of the bench's set-up time.
    The result does not depend on the chunking."""
    coef = [(rng.integers(1, 6, size=2), rng.uniform(0, 2 * np.pi, size=2)) for _ in range(modes)]
    zb = np.zeros_like(x)

    def work(sl):
        acc = np.zeros(sl.stop - sl.start)
        for (kx, ky), ph in coef:
            acc += np.cos(2 * np.pi * kx * x[sl] / lx + ph[0]) * np.cos(2 * np.pi * ky * y[sl] / ly + ph[1])
        zb[sl] = acc

    n, chunk = x.shape[0], 1 << 20
    slices = [slice(a, min(n, a + chunk)) for a in range(0, n, chunk)]
    if len(slices) <= 1:
        for sl in slices:
            work(sl)
    else:
        import os
        from concurrent.futures import ThreadPoolExecutor
        with ThreadPoolExecutor(max_workers=min(16, os.cpu_count() or 1)) as ex:
            list(ex.map(work, slices))
    return amp * zb / modes


def rect_steady(nx=500, ny=250, nsteps=1000):
    """C2: rectangle 100 km x 50 km, nx x ny cells x 2 triangles, steady melt forcing."""
    lx, ly = 100e3, 50e3
    xy, cells = meshgen.rectangle(nx, ny, lx, ly, diagonal="right")
    nv = xy.shape[0]
    x = xy[:, 0]
    f = dict(z_b=np.zeros(nv), z_s=1000.0 * np.sqrt((x + 5e3) / 105e3), G=np.full(nv, 0.05),
             inputs=np.full(nv, 1e-8), storage=np.zeros(nv), b=np.full(nv, 1e-3), N_n=np.full(nv, 0.37e6),
             q=np.zeros((nv, 2)), melt_n=np.zeros(nv))
    t = np.linspace(0.0, 3600.0 * (nsteps - 1), nsteps)
    return Case("rect_steady", xy, cells, f, _left_edge_dofs(nx, ny), 0.37e6, t,
                meta=dict(nx=nx, ny=ny, lx=lx, ly=ly))


def margin_turbulent(nx=2000, ny=1000, lx=200e3, ly=100e3, nsteps=1000, seed=1234, name="margin_turbulent"):
    """C3 (and C4 with nx = ny = 3999, 400 km x 400 km): ice-sheet margin, jittered mesh,
    rough bed, inputs near the margin large enough that |q| exceeds nu/omega (turbulent K)."""
    rng = np.random.default_rng(seed)
    xy, cells = meshgen.rectangle(nx, ny, lx, ly, jitter=0.25, seed=seed, diagonal="right")
    nv = xy.shape[0]
    x, y = xy[:, 0], xy[:, 1]
    z_b = _smooth_bed(x, y, lx, ly, 150.0, rng)
    z_s = 2500.0 * np.sqrt((x + 5e3) / (lx + 5e3))
    z_s = np.maximum(z_s, z_b + 50.0)
    inputs = 3e-8 * np.exp(-x / (0.25 * lx))
    f = dict(z_b=z_b, z_s=z_s, G=np.full(nv, 0.05), inputs=inputs, storage=np.zeros(nv), b=np.full(nv, 1e-3),
             N_n=np.full(nv, 0.37e6), q=np.zeros((nv, 2)), melt_n=np.zeros(nv))
    t = np.linspace(0.0, 3600.0 * (nsteps - 1), nsteps)
    return Case(name, xy, cells, f, _left_edge_dofs(nx, ny), 0.37e6, t, meta=dict(nx=nx, ny=ny, lx=lx, ly=ly))


def dofs16m(nside=4000, nsteps=1000):
    """C4: nside x nside vertices (16M dofs at 4000), same fields as C3 on 400 km x 400 km."""
    scale = nside / 4000.0
    return margin_turbulent(nside - 1, nside - 1, 400e3 * scale, 400e3 * scale, nsteps, name=f"dofs_{nside}x{nside}")


def lakes_fill_drain(nside=8000, nsteps=1000, seed=1234):
    """C5: nside^2 vertices, 8 lake discs (radius 10 km) with storage, inflow pulse."""
    c = margin_turbulent(nside - 1, nside - 1, 800e3 * nside / 8000.0, 800e3 * nside / 8000.0, nsteps, seed,
                         name=f"lakes_{nside}x{nside}")
    lx = c.meta["lx"]
    rng = np.random.default_rng(seed + 1)
    cx = rng.uniform(0.15 * lx, 0.85 * lx, size=8)
    cy = rng.uniform(0.15 * lx, 0.85 * lx, size=8)
    lake = np.zeros(c.n_vert)
    for a, b in zip(cx, cy):
        lake[np.hypot(c.xy[:, 0] - a, c.xy[:, 1] - b) < 10e3 * nside / 8000.0] = 1.0
    c.fields["storage"] = lake
    c.storage_on = True
    c.meta.update(inputs0=c.fields["inputs"].copy(), lake=lake, t_pulse=200 * 3600.0, tau=50 * 3600.0)
    return c


def lake_pulse_inputs(case, t):
    """Time-dependent forcing of C5: inputs0 * (1 + 10 exp(-((t - t_p)/tau)^2)) inside lakes."""
    m = case.meta
    return m["inputs0"] * (1.0 + 10.0 * m["lake"] * np.exp(-(((t - m["t_pulse"]) / m["tau"]) ** 2)))


def cooke2_like(nsteps=87600, seed=2024):
    """C1 surrogate for setups/setup_cooke2.py (the real mesh and datasets are not shipped):
    ~12.3k vertices at 2 km, lake blob with storage, random b_init with a FIXED seed."""
    nx, ny = 110, 110                      # 111 x 111 = 12321 vertices (reference: 12268)
    lx = ly = 2000.0 * nx
    rng = np.random.default_rng(seed)
    xy, cells = meshgen.rectangle(nx, ny, lx, ly, x0=735e3 - 0.0, y0=-1762e3, jitter=0.3, seed=seed, diagonal="random")
    nv = xy.shape[0]
    x, y = xy[:, 0] - 735e3, xy[:, 1] + 1762e3
    z_s = 2122.0 + (2275.0 - 2122.0) * (0.6 * x / lx + 0.4 * y / ly)
    z_b = -535.0 + _smooth_bed(x, y, lx, ly, 405.0, rng)
    lake = (np.hypot(x - 0.5 * lx, y - 0.5 * ly) < 10e3).astype(float)
    potential = 917 * 9.81 * z_s + (1000 - 917) * 9.81 * z_b           # setup_cooke2.py:72
    f = dict(z_b=z_b, z_s=z_s, G=np.full(nv, 0.055), inputs=np.zeros(nv), storage=lake,
             b=0.001 + rng.normal(scale=0.005, size=nv),                 # setup_cooke2.py:66
             N_n=np.full(nv, 3.7e5), q=np.zeros((nv, 2)), melt_n=np.zeros(nv))
    marker = np.abs(potential - potential.min()) < 0.5 * potential.std()  # setup_cooke2.py:80
    t = np.linspace(0.0, 10 * 3.154e7, nsteps)
    c = Case("cooke2_like", xy, cells, f, np.zeros(0, dtype=np.int32), 3.7e5, t, storage_on=True,
             meta=dict(outflow_marker=marker, nx=nx, ny=ny))
    return c


DAY = 86400.0


def diurnal_hydrograph(q_mean, r, knots_per_day=24):
    """Periodic table (times, Q) of max(0, q_mean (1 - r sin 2 pi t / day)) over one day, both ends included."""
    t = np.linspace(0.0, DAY, knots_per_day + 1)
    return t, np.maximum(0.0, q_mean * (1.0 - r * np.sin(2 * np.pi * t / DAY)))


def moulins_like(nx=100, ny=20, n_moulins=60, nsteps=48, seed=7, r=1.2, q_total=60.0):
    """SHMIP-like moulin run (the SHMIP moulin position files are not shipped, so this is seeded, not SHMIP):
    100 km x 20 km ice-sheet margin with the SHMIP square-root surface and a flat bed, outflow at x = 0, a small
    background input and `n_moulins` moulins at seeded positions in 10-90 km.  Each moulin gets a diurnal
    hydrograph max(0, Qbar_k (1 - r sin 2 pi t / day)) tabulated hourly with period one day; the mean discharges
    Qbar_k are seeded and sum to about q_total [m^3/s].  One-hour steps.  meta["moulins"]: (x, y, times, Q) tuples,
    meta["moulin_period"]: the period."""
    lx, ly = 100e3, 20e3
    rng = np.random.default_rng(seed)
    xy, cells = meshgen.rectangle(nx, ny, lx, ly, jitter=0.2, seed=seed, diagonal="alternate")
    nv = xy.shape[0]
    x = xy[:, 0]
    z_s = 6.0 * (np.sqrt(x + 5e3) - np.sqrt(5e3)) + 1.0
    f = dict(z_b=np.zeros(nv), z_s=z_s, G=np.full(nv, 0.05), inputs=np.full(nv, 7.93e-11), storage=np.zeros(nv),
             b=np.full(nv, 0.05), N_n=np.full(nv, 1e5), q=np.zeros((nv, 2)), melt_n=np.zeros(nv))
    mx = rng.uniform(0.1 * lx, 0.9 * lx, size=n_moulins)
    my = rng.uniform(0.05 * ly, 0.95 * ly, size=n_moulins)
    qbar = rng.uniform(0.5, 1.5, size=n_moulins)
    qbar *= q_total / qbar.sum()
    moulins = [(float(a), float(b), *diurnal_hydrograph(q, r)) for a, b, q in zip(mx, my, qbar)]
    t = np.linspace(0.0, 3600.0 * (nsteps - 1), nsteps)
    n_bdry = 917 * 9.81 * z_s.min()            # water at atmospheric pressure under the 1 m thick front
    return Case("moulins_like", xy, cells, f, _left_edge_dofs(nx, ny), n_bdry, t,
                meta=dict(nx=nx, ny=ny, lx=lx, ly=ly, moulins=moulins, moulin_period=DAY))


def apply_case(model, case):
    """Upload a Case into a capi.Model and perform solvers.py:48 (N <- N_n)."""
    for k in ("z_b", "z_s", "G", "inputs", "storage", "b", "N_n", "melt_n"):
        model.set_field(k, case.fields[k])
    model.set_flux(case.fields["q"])
    bc = case.bc_dofs
    if bc.size == 0 and "outflow_marker" in case.meta:
        bc = model.locate_dirichlet(case.meta["outflow_marker"])
    model.set_dirichlet(bc, case.N_bdry)
    model.start()
    return model
