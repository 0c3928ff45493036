"""CPU reference of the water-budget record (test infrastructure, like oracle/): the columns of enum shakti_diag
(include/shakti_b200.h) at the current state of a ShaktiOracle, every integral restated per quadrature point with
the oracle's own table, in the style of ShaktiOracle.element_FJ.  outflow / imbalance: the unconstrained element
residual (no lifting, no Dirichlet replacement) summed onto Dirichlet / other vertices."""
import numpy as np


def oracle_diagnostics(o, dt):
    """Record of ShaktiOracle `o` at its current N (with its lagged b, q, melt_n, N_n) -> dict keyed like
    capi.DIAGNOSTICS (newton_its is 0, residual is ||F|| of the Dirichlet-handled assembly)."""
    p = o.p
    c = o.cells
    N = o.N
    Fe, _ = o.element_FJ(dt, N, want_J=False)
    isbc = np.zeros(o.nv, dtype=bool)
    isbc[o.bc_dofs] = True
    bce = isbc[c]
    F, _ = o.assemble(dt, want_J=False)
    gh = o._cell_grad(o.head(N))
    gb = o._cell_grad(o.b)
    gm = o._cell_grad(o.melt_n)
    gb2 = np.einsum("ek,ek->e", gb, gb)
    gmgb = np.einsum("ek,ek->e", gm, gb)
    Nc, Nnc, bc = N[c], o.N_n[c], o.b[c]
    qc, Gc, mc = o.q[c], o.G[c], o.melt_n[c]
    sc, ic = o.storage[c], o.inputs[c]
    s = dict(area=0.0, water_volume=0.0, input=0.0, melt=0.0, closure=0.0, storage=0.0, intN=0.0)
    for (xi, eta), w in zip(o.qpts, o.qwts):
        lam = np.array([1.0 - xi - eta, xi, eta])
        wd = w * o.detabs
        bq, Nq, Nnq = bc @ lam, Nc @ lam, Nnc @ lam
        Gq, mq, sq, iq = Gc @ lam, mc @ lam, sc @ lam, ic @ lam
        qq = np.einsum("eak,a->ek", qc, lam)
        qgh = np.einsum("ek,ek->e", qq, gh)
        m0 = (Gq - p.rho_w * p.g * qgh) / p.Lh               # constitutive.py:25
        mdiff = (gb2 * mq + bq * gmgb) / (1 + gb2)           # constitutive.py:26
        s["area"] += wd.sum()
        s["water_volume"] += (wd * bq).sum()
        s["input"] += (wd * iq).sum()
        s["melt"] += (wd * (m0 + mdiff)).sum()
        s["closure"] += (wd * p.A * bq * Nq * np.abs(Nq) ** (p.n - 1)).sum()
        s["storage"] += (wd * sq * (Nq - Nnq)).sum() / (p.rho_w * p.g * dt)
        s["intN"] += (wd * Nq).sum()
    intN = s.pop("intN")
    s = {k: float(v) for k, v in s.items()}
    return dict(dt=float(dt), newton_its=0.0, residual=float(np.linalg.norm(F)), **s,
                outflow=float(-Fe[bce].sum()), imbalance=float(Fe[~bce].sum()), N_mean=float(intN / s["area"]),
                N_min=float(N.min()), N_max=float(N.max()), b_max=float(o.b.max()))
