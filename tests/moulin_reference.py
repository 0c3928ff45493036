"""CPU reference of moulins (test infrastructure, like oracle/): the oracle with a model clock and point sources
F_i -= sum_{k: v_k = i} Q_k(t) after the assembly (include/shakti_b200.h, shakti_set_moulins).  The hydrograph is
restated with numpy's own linear interpolation; oracle/ itself stays unchanged."""
import numpy as np

from oracle.shakti_oracle import ShaktiOracle


def hydrograph(t_knots, q_knots, t, period=0.0):
    """Q(t): np.interp of the knots (constant outside them), after wrapping t into [t_0, t_0 + period)."""
    tk = np.asarray(t_knots, dtype=np.float64)
    t = np.asarray(t, dtype=np.float64)
    if period > 0:
        t = tk[0] + np.mod(t - tk[0], period)
    return np.interp(t, tk, np.asarray(q_knots, dtype=np.float64))


class MoulinOracle(ShaktiOracle):
    """ShaktiOracle with moulins: ``moulins`` is a list of (vertex, times, discharges); ``t`` the model clock.
    A solve with step dt is forced at t + dt and ``step`` advances t by dt, like the library."""

    def __init__(self, *args, **kw):
        super().__init__(*args, **kw)
        self.t = 0.0
        self.moulins, self.period = [], 0.0

    def set_moulins(self, moulins, period=0.0):
        self.moulins, self.period = list(moulins), float(period)

    def moulin_discharge(self, t):
        return np.array([hydrograph(tk, qk, t, self.period) for _, tk, qk in self.moulins])

    def moulin_source(self, t):
        """Nodal vector of the moulin discharge at t (duplicates summed in the order given)."""
        s = np.zeros(self.nv)
        for (v, _, _), q in zip(self.moulins, self.moulin_discharge(t)):
            s[v] += q
        return s

    def assemble(self, dt, N=None, want_J=True):
        F, vals = super().assemble(dt, N, want_J)
        if self.moulins:
            F = F - self.moulin_source(self.t + dt)
        return F, vals

    def step(self, dt):
        out = super().step(dt)
        self.t += dt
        return out


def moulin_diagnostics(o, dt):
    """Water-budget record of MoulinOracle `o` (budget_reference.oracle_diagnostics): the moulin discharge at o.t + dt
    is part of the input, and the imbalance -- the sum of F~ over the non-Dirichlet rows -- includes the moulin rows."""
    from budget_reference import oracle_diagnostics
    d = oracle_diagnostics(o, dt)
    q = float(o.moulin_discharge(o.t + dt).sum()) if o.moulins else 0.0
    d["input"] += q
    d["imbalance"] -= q
    return d
