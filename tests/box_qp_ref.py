"""Optimality of a box-constrained QP step, for the tests of the IK solve (a helper module, not a test file).

    minimise f(x) = 1/2 x'Ax + b'x   subject to   lo <= x <= hi          (A symmetric positive definite)

`kkt_certificate` judges a given x by the first-order conditions alone, so it needs no second solver and no assumption
about how x was found: it can be run on the float64 A, b and delta the IK step returns.  `reference_box_qp` is an
independent solve (scipy's bounded-variable least squares on the Cholesky factor of A), used to compare objective values
where A is ill-conditioned and x itself is not well determined.

Column layout of the IK unknowns (the reference layout of smplpp_ik_step's A / b / delta outputs):
    theta (theta_dim) | phi (2 n, two per task) | beta (10, only with optimize_beta)
"""
from __future__ import annotations

import numpy as np

KKT_TOL = 1e-10      # gradient / multiplier violations allowed, relative to the problem scale
FEAS_TOL = 1e-12     # bound violations allowed, relative to the bound


def problem_scale(A, b, x) -> float:
    """s = ||A||_max * max(1, ||x||_inf) + ||b||_inf: the size of the terms that make up the gradient A x + b."""
    return float(np.abs(A).max(initial=0.0) * max(1.0, np.abs(x).max(initial=0.0)) + np.abs(b).max(initial=0.0))


def objective(A, b, x) -> float:
    A, b, x = (np.asarray(v, np.float64) for v in (A, b, x))
    return float(0.5 * x @ (A @ x) + b @ x)


def ik_blocks(theta_dim: int, n: int, dim: int) -> dict:
    """Column blocks of the reference layout: {name: (first, end)}."""
    return {"theta": (0, theta_dim), "phi": (theta_dim, theta_dim + 2 * n), "beta": (theta_dim + 2 * n, dim)}


def _block_of(i, blocks):
    if not blocks:
        return "x"
    for name, (a, e) in blocks.items():
        if a <= i < e:
            return name
    return "?"


def kkt_certificate(A, b, x, lo, hi, blocks=None, tol=None):
    """First-order optimality of x for min 1/2 x'Ax + b'x over lo <= x <= hi, with g = A x + b in float64:
      feasibility         lo - 1e-12 |lo| <= x <= hi + 1e-12 |hi|;
      interior unknowns   |g_i| <= tol * s;
      at the upper bound  g_i <= tol * s         (x_i >= hi_i; the multiplier -g_i is >= 0);
      at the lower bound  g_i >= -tol * s        (x_i <= lo_i);
      lo_i == hi_i        no sign condition (the unknown is pinned).
    s = problem_scale(A, b, x).  An unknown counts as at its bound only when it equals the bound (or lies beyond it
    within the feasibility tolerance): a solver that leaves an active unknown a hair inside its box has to make its
    gradient vanish there.
    Returns (ok, report); report holds the scale, the worst ratio |violation| / s, the worst unknown, its column block
    (`blocks`, see ik_blocks) and its kind, and the number of unknowns at each bound."""
    tol = KKT_TOL if tol is None else tol
    A, b, x, lo, hi = (np.asarray(v, np.float64) for v in (A, b, x, lo, hi))
    g = A @ x + b
    s = problem_scale(A, b, x)
    pinned = lo == hi
    at_hi = ~pinned & np.isfinite(hi) & (x >= hi)
    at_lo = ~pinned & np.isfinite(lo) & (x <= lo)
    interior = ~pinned & ~at_hi & ~at_lo
    feas = np.maximum(np.where(np.isfinite(lo), lo - FEAS_TOL * np.abs(lo) - x, 0.0),
                      np.where(np.isfinite(hi), x - hi - FEAS_TOL * np.abs(hi), 0.0))
    viol = np.zeros_like(x)
    viol[interior] = np.abs(g[interior])
    viol[at_hi] = np.maximum(g[at_hi], 0.0)
    viol[at_lo] = np.maximum(-g[at_lo], 0.0)
    ratio = viol / s if s > 0 else viol
    kind = np.where(pinned, "pinned", np.where(at_hi, "upper", np.where(at_lo, "lower", "interior")))
    report = dict(scale=s, worst_ratio=float(ratio.max(initial=0.0)), n_upper=int(at_hi.sum()),
                  n_lower=int(at_lo.sum()), n_pinned=int(pinned.sum()), worst=None)
    ok = True
    if feas.size and feas.max() > 0.0:
        k = int(np.argmax(feas))
        ok = False
        report["worst"] = "unknown %d (%s) outside [%.17g, %.17g]: x = %.17g" % (k, _block_of(k, blocks), lo[k], hi[k], x[k])
    elif ratio.size:
        k = int(np.argmax(ratio))
        if ratio[k] > tol:
            ok = False
        report["worst"] = "unknown %d (%s, %s): x = %.17g, g = %.3e, |violation| / s = %.3e" % (
            k, _block_of(k, blocks), kind[k], x[k], g[k], ratio[k])
    return ok, report


def reference_box_qp(A, b, lo, hi) -> np.ndarray:
    """Independent float64 solve: with A = R'R, minimise 1/2 ||R x + R^-T b||^2 (= f(x) + const) over the box by
    scipy.optimize.lsq_linear(method="bvls").  Unknowns with lo == hi are substituted before the solve (bvls wants
    lo < hi); unbounded unknowns get +-inf."""
    from scipy.linalg import cho_factor, solve_triangular
    from scipy.optimize import lsq_linear
    A, b, lo, hi = (np.asarray(v, np.float64) for v in (A, b, lo, hi))
    x = np.zeros_like(b)
    pinned = lo == hi
    x[pinned] = lo[pinned]
    free = np.nonzero(~pinned)[0]
    if free.size == 0:
        return x
    Aff = A[np.ix_(free, free)]
    bf = b[free] + A[np.ix_(free, np.nonzero(pinned)[0])] @ x[pinned]
    R = np.triu(cho_factor(Aff, lower=False)[0])
    rhs = -solve_triangular(R, bf, trans="T")
    res = lsq_linear(R, rhs, bounds=(lo[free], hi[free]), method="bvls", tol=1e-15, lsq_solver="exact",
                     max_iter=50 * free.size + 100)
    if res.status < 0 or res.status == 0:
        raise RuntimeError("bvls did not converge (status %d: %s)" % (res.status, res.message))
    xf = np.clip(res.x, lo[free], hi[free])
    # bvls can leave a bound-active unknown a rounding step inside its box; put it on the bound it reports active
    xf = np.where(res.active_mask > 0, hi[free], np.where(res.active_mask < 0, lo[free], xf))
    x[free] = xf
    return x


def objective_gap_tol(A, b, x, rel=1e-12) -> float:
    """The allowed excess of f(x) over the reference optimum: rel * (|f(x)| + s ||x||_inf)."""
    return rel * (abs(objective(A, b, x)) + problem_scale(A, b, x) * float(np.abs(x).max(initial=0.0)))


def ik_bounds(opts: dict, n: int, dim_ref: int, theta_dim: int):
    """lo, hi of the IK step's unknowns in the reference layout, from the options as the step reads them:
      phi is bounded by +-phi_limit when enable_phi and phi_limit > 0; otherwise the phi columns do not exist and delta's
          phi entries are exactly 0 (lo = hi = 0);
      beta (optimize_beta) is bounded by +-delta_beta_limit;
      enable_qp = 0 bounds nothing (existing phi / beta columns get +-inf).
    The limits are float32 options, widened exactly like the kernels widen them."""
    lo = np.full(dim_ref, -np.inf)
    hi = np.full(dim_ref, np.inf)
    qp = bool(opts.get("enable_qp", 1))
    phi_limit = float(np.float32(opts.get("phi_limit", 0.0)))
    ph = slice(theta_dim, theta_dim + 2 * n)
    if opts.get("enable_phi") and phi_limit > 0.0:
        if qp:
            lo[ph], hi[ph] = -phi_limit, phi_limit
    else:
        lo[ph], hi[ph] = 0.0, 0.0
    if opts.get("optimize_beta"):
        assert dim_ref == theta_dim + 2 * n + 10
        if qp:
            lim = float(np.float32(opts.get("delta_beta_limit", 0.5)))
            lo[theta_dim + 2 * n:], hi[theta_dim + 2 * n:] = -lim, lim
    else:
        assert dim_ref == theta_dim + 2 * n
    return lo, hi


def multipliers(A, b, x, lo, hi) -> np.ndarray:
    """The bound multiplier of every unknown (0 where interior or pinned): -g_i at the upper bound, g_i at the lower one."""
    A, b, x, lo, hi = (np.asarray(v, np.float64) for v in (A, b, x, lo, hi))
    g = A @ x + b
    pinned = lo == hi
    lam = np.zeros_like(x)
    up = ~pinned & np.isfinite(hi) & (x >= hi)
    dn = ~pinned & np.isfinite(lo) & (x <= lo)
    lam[up] = -g[up]
    lam[dn] = g[dn]
    return lam


def active_set(x, lo, hi) -> np.ndarray:
    """+1 at the upper bound, -1 at the lower one, 0 interior or pinned."""
    pinned = lo == hi
    return np.where(~pinned & np.isfinite(hi) & (x >= hi), 1, np.where(~pinned & np.isfinite(lo) & (x <= lo), -1, 0))
