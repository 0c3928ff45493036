"""Shared synthetic cases for the parity tests (seeded; small enough for the oracle)."""
import numpy as np

from oracle.shakti_oracle import ShaktiOracle, dirichlet_dofs
from shakti_b200 import meshgen


def make_case(nx=24, ny=16, seed=0, scramble=True, storage=True, turbulent=True, neg_b=False, diagonal="random"):
    """Jittered rectangle 100 km x 50 km with rough, fully populated fields (every term of the
    residual active).  Returns (xy, cells, fields dict, bc_dofs, N_bdry)."""
    xy, cells = meshgen.rectangle(nx, ny, 100e3, 50e3, jitter=0.25, seed=seed + 11, diagonal=diagonal)
    if scramble:
        xy, cells = meshgen.scramble(xy, cells, seed=seed + 5)
    return case_on(xy, cells, seed, storage=storage, turbulent=turbulent, neg_b=neg_b)


def case_on(xy, cells, seed=0, storage=True, turbulent=True, neg_b=False):
    """The fields of make_case on any mesh of the 100 km x 50 km domain: storage on the disc of radius 15 km around
    the centre, Dirichlet dofs on x = 0.  Returns (xy, cells, fields dict, bc_dofs, N_bdry)."""
    nv = xy.shape[0]
    x, y = xy[:, 0], xy[:, 1]
    rng = np.random.default_rng(seed)
    f = {}
    f["z_b"] = 50 * np.cos(x / 2e4) * np.sin(y / 1.5e4)
    f["z_s"] = 1000 * np.sqrt((x + 5e3) / 105e3)
    f["G"] = 0.05 + 0.01 * rng.random(nv)
    f["inputs"] = 1e-8 * (1 + rng.random(nv))
    f["storage"] = (np.hypot(x - 5e4, y - 2.5e4) < 1.5e4).astype(float) if storage else np.zeros(nv)
    f["b"] = 1e-3 * (1 + 0.5 * rng.random(nv))
    if neg_b:
        f["b"] = 0.001 + rng.normal(scale=0.005, size=nv)      # setup_cooke2.py:66 (seeded here)
    f["N_n"] = 0.37e6 * (1 + 0.05 * rng.random(nv))
    qs = 2e-3 if turbulent else 1e-6
    f["q"] = qs * rng.standard_normal((nv, 2))
    f["melt_n"] = 1e-6 * rng.random(nv)
    N_bdry = 0.37e6
    bc = dirichlet_dofs(xy, cells, lambda X: np.isclose(X[0], 0.0))
    return xy, cells, f, bc, N_bdry


def make_oracle(xy, cells, f, bc, N_bdry, **kw):
    o = ShaktiOracle(xy, cells, **kw)
    for k in ("z_b", "z_s", "G", "inputs", "storage", "b", "N_n", "melt_n"):
        getattr(o, k)[:] = f[k]
    o.q[:] = f["q"]
    o.set_dirichlet(bc, N_bdry)
    o.start()
    return o


def make_model(xy, cells, f, bc, N_bdry, **opt):
    from shakti_b200 import capi
    m = capi.Model(xy, cells, **opt)
    for k in ("z_b", "z_s", "G", "inputs", "storage", "b", "N_n", "melt_n"):
        m.set_field(k, f[k])
    m.set_flux(f["q"])
    m.set_dirichlet(bc, N_bdry)
    m.start()
    return m


def relinf(a, b):
    return float(np.max(np.abs(np.asarray(a) - np.asarray(b))) / max(np.max(np.abs(b)), 1e-300))


class OracleStepper:
    """Adapter of the CPU oracle for shakti_b200.golden.check."""

    def __init__(self, dump, **kw):
        from oracle.shakti_oracle import Params
        from shakti_b200.golden import FIELDS
        o = ShaktiOracle(dump.xy, dump.cells, params=Params(**dump.meta["params"]), quad=dump.quad, **kw)
        for k in FIELDS:
            getattr(o, k)[:] = dump.initial[k]
        o.q[:] = dump.initial["q"]
        o.set_dirichlet(dump.bc_dofs, dump.N_bdry)
        o.start()
        self.o = o

    def assemble(self, dt):
        F, v = self.o.assemble(dt)
        return F, (self.o.rowptr, self.o.col, v)

    def step(self, dt):
        return self.o.step(dt)[0]

    def state(self):
        return dict(N=self.o.N, b=self.o.b, q=self.o.q, melt_n=self.o.melt_n)


