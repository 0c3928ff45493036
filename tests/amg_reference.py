"""Float64 reference of the smoothed-aggregation AMG of csrc/amg.cu (test infrastructure, like budget_reference.py).

It restates coarsen_level, numeric_level and vcycle with scipy, one rank:

- aggregates: shakti_host_amg_aggregate (the library's own greedy aggregation, CPU-checked against
  tools/amg_prototype.py) on the reference's A_l, strength threshold theta 0.5^l, Dirichlet rows excluded on level 0;
- P = diag(keep) (I - omega D^-1 A) T, the columns of excluded vertices dropped; R = P^T (own block of one rank);
  A_{l+1} = R (A P).  Patterns come from products of matrices of ones (scipy drops the exact zeros of a product,
  the library keeps every structural entry);
- the Chebyshev bound max_i |dinv_i| sum_j |a_ij| and the coefficient recurrence of amg_cheby_coef_kernel, in its order
  of operations (a bound that is not positive and finite gives 2.0);
- the V-cycle: zero-guess first step, Chebyshev or damped-Jacobi sweeps, residual, restriction, the coarsest level by
  its dense inverse (<= 1024 rows) or 8 Chebyshev sweeps, prolongation, post-smoothing whose sweep 0 has c1 = 0.

Switches: with_fine() gives the lagged hierarchy (level 0 on the current J, P, R and the coarse levels from the J of
the last full refresh); with_half() replaces a level's operator by D f16(f32(D^-1 A)).  The comparisons with the
library's exports are plain functions of the exports, so that a CPU test can feed them the reference's own.
"""
from dataclasses import dataclass, replace

import numpy as np
import scipy.sparse as sp

DENSE_MAX = 1024          # the coarsest level is inverted densely up to this many rows (build_hierarchy)
COARSEST_SWEEPS = 8       # Chebyshev sweeps on a coarsest level that is not dense
STALL = 0.85              # coarsening stops when a level keeps more than this share of its rows


@dataclass(frozen=True)
class Options:
    """The AMG options of shakti_options (shakti_default_options' values)."""
    max_levels: int = 12
    coarse_size: int = 256
    presmooth: int = 2
    postsmooth: int = 2
    smoother: str = "chebyshev"       # or "jacobi"
    smoother_omega: float = 0.67
    prolong_omega: float = 0.67
    theta: float = 0.08
    ratio: float = 5.0

    @staticmethod
    def of(opt):
        """From a capi.Options structure."""
        return Options(opt.amg_max_levels, opt.amg_coarse_size, opt.amg_presmooth, opt.amg_postsmooth,
                       "chebyshev" if opt.amg_smoother == 1 else "jacobi", opt.amg_smoother_omega, opt.amg_prolong_omega,
                       opt.amg_strength_theta, opt.amg_cheby_ratio)

    @property
    def coef_sweeps(self):
        return max(self.presmooth, self.postsmooth, COARSEST_SWEEPS)


@dataclass
class Level:
    A: sp.csr_matrix
    dinv: np.ndarray
    coef: np.ndarray = None       # Chebyshev table (coef_layout); None with the Jacobi smoother
    P: sp.csr_matrix = None
    R: sp.csr_matrix = None
    last: bool = False
    inverse: np.ndarray = None    # dense inverse of a coarsest level of <= DENSE_MAX rows


# ------------------------------------------------------------------------------------------------ building blocks
def ones(A):
    """The stored pattern of A with every value 1 (explicit zeros included)."""
    A = sp.csr_matrix(A)
    return sp.csr_matrix((np.ones(A.indices.size), A.indices.copy(), A.indptr.copy()), shape=A.shape)


def on_pattern(S, V):
    """CSR with S's pattern (sorted) and V's values there (0 where V has none)."""
    S = sp.csr_matrix(S)
    S.sum_duplicates()
    S.sort_indices()
    rows = np.repeat(np.arange(S.shape[0]), np.diff(S.indptr))
    vals = np.asarray(sp.csr_matrix(V)[rows, S.indices]).ravel() if S.nnz else np.zeros(0)
    return sp.csr_matrix((vals.astype(np.float64), S.indices.copy(), S.indptr.copy()), shape=S.shape)


def dinv_of(A):
    d = A.diagonal()
    out = np.zeros_like(d)
    np.divide(1.0, d, out=out, where=d != 0.0)
    return out


def gershgorin(A, dinv):
    """max_i |dinv_i| sum_j |a_ij| (amg_gershgorin_kernel)."""
    if A.shape[0] == 0:
        return 0.0
    return float(np.max(np.abs(dinv) * np.asarray(abs(A).sum(axis=1)).ravel()))


def cheby_coef(bound, ratio, sweeps):
    """amg_cheby_coef_kernel for one level: [1/theta, 0, then (c1, c2) of sweep k at 2 + 2k], same operations in the
    same order (Python floats are IEEE doubles without contraction)."""
    hi = float(bound) if (bound > 0.0 and np.isfinite(bound)) else 2.0
    lo = hi / ratio
    theta, delta = 0.5 * (hi + lo), 0.5 * (hi - lo)
    sigma = theta / delta
    rho = 1.0 / sigma
    c = np.zeros(2 + 2 * sweeps)
    c[0] = 1.0 / theta
    c[2], c[3] = 0.0, c[0]
    for k in range(1, sweeps):
        rho_n = 1.0 / (2.0 * sigma - rho)
        c[2 + 2 * k] = rho_n * rho
        c[3 + 2 * k] = (2.0 * rho_n) / delta
        rho = rho_n
    return c


def aggregates(A, level, exclude, theta):
    """Aggregates of level `level` (exclude: Dirichlet rows, used on level 0 only) -> (agg, count)."""
    from shakti_b200 import capi
    A = sp.csr_matrix(A)
    A.sort_indices()
    return capi.host_amg_aggregate(A, theta * 0.5 ** level, exclude if level == 0 else None)


def prolongator(A, dinv, agg, n_agg, omega):
    """P = diag(keep) (I - omega D^-1 A) T on the library's pattern (numeric_level / amg_prolongator_kernel)."""
    n = A.shape[0]
    keep = agg >= 0
    rows = np.nonzero(keep)[0]
    T = sp.csr_matrix((np.ones(rows.size), (rows, agg[rows])), shape=(n, n_agg))
    K = sp.diags(keep.astype(np.float64))
    S = K @ (ones(A) + sp.eye(n, format="csr")) @ T
    V = K @ ((sp.eye(n, format="csr") - sp.diags(omega * dinv) @ A) @ T)
    return on_pattern(S, V)


def galerkin(R, A, P):
    """A_{l+1} = R (A P) on the pattern of the library's symbolic products, and the entrywise summation bound
    (|R| |A| |P|)_ij on the same pattern."""
    S = ones(R) @ (ones(A) @ ones(P))
    return on_pattern(S, R @ (A @ P)), on_pattern(S, abs(R) @ (abs(A) @ abs(P)))


def smoother_coef(A, dinv, opt, bound=None):
    if opt.smoother != "chebyshev":
        return None
    # one spare sweep: the shifted-coefficient mutation reads sweep k + 1
    return cheby_coef(gershgorin(A, dinv) if bound is None else bound, opt.ratio, opt.coef_sweeps + 1)


# ------------------------------------------------------------------------------------------------ hierarchy
def build(J, exclude, opt=Options()):
    """The hierarchy of the fine matrix J (CSR, sorted) with Dirichlet rows `exclude` (bool, level 0)."""
    J = sp.csr_matrix(J)
    J.sort_indices()
    levels = []
    A = J
    for l in range(opt.max_levels):
        n = A.shape[0]
        dinv = dinv_of(A)
        L = Level(A, dinv, smoother_coef(A, dinv, opt))
        levels.append(L)
        stop = n <= opt.coarse_size or l + 1 >= opt.max_levels
        if not stop:
            agg, na = aggregates(A, l, exclude, opt.theta)
            stop = na <= 0 or na > STALL * n
        if stop:
            L.last = True
            if 0 < n <= DENSE_MAX:
                L.inverse = np.linalg.inv(A.toarray())
            break
        L.P = prolongator(A, dinv, agg, na, opt.prolong_omega)
        L.R = sp.csr_matrix(L.P.T)
        L.R.sort_indices()
        A = galerkin(L.R, A, L.P)[0]
    return Hierarchy(levels, opt)


@dataclass
class Hierarchy:
    levels: list
    opt: Options

    def with_fine(self, J):
        """The lagged hierarchy after a fine-smoother refresh: level 0 on J (diagonal and bound from J), everything
        else kept.  A one-level hierarchy keeps its dense inverse (it is not refreshed)."""
        J = sp.csr_matrix(J)
        J.sort_indices()
        L0 = self.levels[0]
        dinv = dinv_of(J)
        coef = L0.coef
        if coef is not None and not (L0.last and L0.inverse is not None):
            coef = smoother_coef(J, dinv, self.opt)
        return Hierarchy([replace(L0, A=J, dinv=dinv, coef=coef)] + self.levels[1:], self.opt)

    def with_half(self, levels):
        """Levels `levels` run on the half-precision copy of D^-1 A: operator D f16(f32(D^-1 A))."""
        out = list(self.levels)
        for l in levels:
            L = out[l]
            A = sp.csr_matrix(L.A)
            rows = np.repeat(np.arange(A.shape[0]), np.diff(A.indptr))
            h = (L.dinv[rows] * A.data).astype(np.float32).astype(np.float16).astype(np.float64)
            d = np.zeros_like(L.dinv)
            np.divide(1.0, L.dinv, out=d, where=L.dinv != 0.0)
            out[l] = replace(L, A=sp.csr_matrix((d[rows] * h, A.indices, A.indptr), shape=A.shape))
        return Hierarchy(out, self.opt)

    def with_options(self, **kw):
        return replace(self, opt=replace(self.opt, **kw))


# ------------------------------------------------------------------------------------------------ V-cycle
# Mutations (discrimination checks: each is a plausible kernel bug that a right tolerance must see):
#   "drop_slice"  the smoother and residual of level 1 skip its last 32-row slice (rows keep their old values)
#   "shift_post"  post-smoothing sweep k uses the coefficients of sweep k + 1
#   "stale_d"     post-smoothing sweep 0 uses c1 of sweep 1 on the d left by the pre-smoothing
#   "no_coarse"   no coarse-grid correction below level 1
MUTATIONS = ("drop_slice", "shift_post", "stale_d", "no_coarse")


def vcycle(H, b, mutations=()):
    """z = M^-1 b: one V-cycle from a zero guess."""
    return _cycle(H, 0, np.asarray(b, dtype=np.float64), frozenset(mutations))


def _last_slice(n):
    return np.arange(32 * ((n - 1) // 32), n) if n > 0 else np.zeros(0, int)


def _cycle(H, l, b, mut):
    L = H.levels[l]
    if L.last:
        if L.inverse is not None:
            return L.inverse @ b
        return _smooth(H, l, b, None, COARSEST_SWEEPS, mut)[0]
    x, d = _smooth(H, l, b, None, H.opt.presmooth, mut)
    r = b - L.A @ x
    if "drop_slice" in mut and l == 1:
        r[_last_slice(L.A.shape[0])] = 0.0
    xc = np.zeros(L.P.shape[1]) if ("no_coarse" in mut and l == 1) else _cycle(H, l + 1, L.R @ r, mut)
    x = x + L.P @ xc
    return _smooth(H, l, b, x, H.opt.postsmooth, mut, d=d, post=True)[0]


def _smooth(H, l, b, x, sweeps, mut, d=None, post=False):
    """`sweeps` steps on A x = b from x (None: zero guess) -> (x, d)."""
    L, opt = H.levels[l], H.opt
    n = L.A.shape[0]
    skip = _last_slice(n) if ("drop_slice" in mut and l == 1) else None
    if x is None and sweeps <= 0:
        return np.zeros(n), d
    k0 = 0
    if opt.smoother != "chebyshev":
        om = opt.smoother_omega
        if x is None:
            x, k0 = om * L.dinv * b, 1
        for _ in range(k0, sweeps):
            xn = x + om * L.dinv * (b - L.A @ x)
            if skip is not None:
                xn[skip] = x[skip]
            x = xn
        return x, None
    c = L.coef
    if x is None:
        d = L.dinv * b * c[0]
        x, k0 = d.copy(), 1
    for k in range(k0, sweeps):
        kk = k + 1 if (post and "shift_post" in mut) else k
        c1, c2 = c[2 + 2 * kk], c[3 + 2 * kk]
        if post and k == 0 and "stale_d" in mut:
            c1 = c[4]
        r = L.dinv * (b - L.A @ x)
        dn = (c1 * d if (d is not None and c1 != 0.0) else 0.0) + c2 * r
        xn = x + dn
        if skip is not None:
            dn[skip] = d[skip] if d is not None else 0.0
            xn[skip] = x[skip]
        d, x = dn, xn
    return x, d


# ------------------------------------------------------------------------------------------------ comparisons
def exports_of(H):
    """What the library exports per level (Model.amg_matrix / amg_vectors), made from the reference itself."""
    out = []
    for L in H.levels:
        e = dict(A=L.A, dinv=L.dinv, last=L.last)
        if L.coef is not None:
            e["coef"] = L.coef[: 2 + 2 * H.opt.coef_sweeps]
        if not L.last:
            e["P"], e["R"] = L.P, L.R
        out.append(e)
    return out


def same_csr(a, b, values=True):
    a, b = sp.csr_matrix(a), sp.csr_matrix(b)
    return (a.shape == b.shape and np.array_equal(a.indptr, b.indptr) and np.array_equal(a.indices, b.indices)
            and (not values or np.array_equal(a.data, b.data)))


def entry_distance(dev, ref, scale):
    """max_ij |dev - ref| / scale_ij over the common pattern (scale 0: the entries must be equal)."""
    diff = np.abs(sp.csr_matrix(dev).data - sp.csr_matrix(ref).data)
    s = sp.csr_matrix(scale).data
    if np.any(diff[s == 0.0] != 0.0):
        return np.inf
    return float(np.max(diff[s > 0] / s[s > 0], initial=0.0))


def row_max(P):
    P = sp.csr_matrix(P)
    rows = np.repeat(np.arange(P.shape[0]), np.diff(P.indptr))
    m = np.zeros(P.shape[0])
    np.maximum.at(m, rows, np.abs(P.data))
    return sp.csr_matrix((m[rows], P.indices, P.indptr), shape=P.shape)


def compare_levels(exp, exclude, opt=Options()):
    """Check every level of the exports `exp` (list of dicts A, P, R, dinv, coef, last) against the reference made
    from the exports' own inputs of that level, so that each distance measures one step only:
    P from A_l (aggregates of A_l), A_{l+1} from R_l, A_l, P_l; dinv from A_l; coefficients from A_l and dinv_l.
    -> dict of distances (P: relative to the row's largest |p|; galerkin: relative to (|R||A||P|)_ij; coef: relative)
    and exactness flags."""
    res = dict(P=0.0, galerkin=0.0, coef=0.0, patterns=True, dinv_exact=True, R_exact=True)
    for l, e in enumerate(exp):
        A = sp.csr_matrix(e["A"])
        res["dinv_exact"] &= bool(np.array_equal(e["dinv"], dinv_of(A)))
        if "coef" in e and opt.smoother == "chebyshev":
            ref = cheby_coef(gershgorin(A, e["dinv"]), opt.ratio, opt.coef_sweeps)
            res["coef"] = max(res["coef"], float(np.max(np.abs(e["coef"] - ref)) / np.max(np.abs(ref))))
        if e["last"]:
            continue
        agg, na = aggregates(A, l, exclude, opt.theta)
        Pref = prolongator(A, dinv_of(A), agg, na, opt.prolong_omega)
        if not same_csr(e["P"], Pref, values=False):
            res["patterns"] = False
            continue
        res["P"] = max(res["P"], entry_distance(e["P"], Pref, row_max(Pref)))
        Rt = sp.csr_matrix(sp.csr_matrix(e["P"]).T)
        Rt.sort_indices()
        res["R_exact"] &= same_csr(e["R"], Rt)
        C, bound = galerkin(sp.csr_matrix(e["R"]), A, sp.csr_matrix(e["P"]))
        if not same_csr(exp[l + 1]["A"], C, values=False):
            res["patterns"] = False
            continue
        res["galerkin"] = max(res["galerkin"], entry_distance(exp[l + 1]["A"], C, bound))
    return res


def rel_inf(z, ref):
    return float(np.max(np.abs(np.asarray(z) - ref)) / max(np.max(np.abs(ref)), 1e-300))


def discrimination(H, b, tol, J, exclude):
    """How far each mutation of the reference moves z, in units of tol (relative infinity norm): all must be >= 10.
    "omega" rebuilds the hierarchy from J with prolong_omega 0.66 instead of 0.67."""
    z = vcycle(H, b)
    out = {m: rel_inf(vcycle(H, b, (m,)), z) / tol for m in MUTATIONS}
    out["omega"] = rel_inf(vcycle(build(J, exclude, replace(H.opt, prolong_omega=0.66)), b), z) / tol
    return out
