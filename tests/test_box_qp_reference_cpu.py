"""The box-QP optimality certificate of tests/box_qp_ref.py on random strictly convex problems shaped like the IK step's
(no GPU).

It must accept what two independent float64 solvers return (scipy's bvls, and the oracle's primal active set
`solve_box_qp`, the iteration the CUDA kernels restate), and reject the failures a bounded solve can have: an active
unknown left just inside its box, a bound taken on the wrong side, the unconstrained step clipped to the box.  The two
solvers must agree on the optimal objective.

Problems: D in {10, 44, 85, 136, 239} (the IK sizes from VPoser-only to a body stage with 82 tasks), the first third of
the unknowns unbounded like theta, A = J'J + (1e-3 + ||e||^2) I like the step's damping, J scaled by 1e-3, 1 and 1e3,
and limits that bind nothing, about half, nearly everything (1e-4), or pin the bounded unknowns at 0; plus degenerate
problems with one unknown's optimum exactly on its bound (zero multiplier).
"""
from __future__ import annotations

import numpy as np
import pytest

import box_qp_ref as q

SIZES = (10, 44, 85, 136, 239)
SCALES = (1e-3, 1.0, 1e3)
KINDS = ("none", "half", "all", "zero", "degenerate_free", "degenerate_mixed")
CASES = [(d, s, k) for d in SIZES for s in SCALES for k in KINDS]


def make_problem(D, scale, kind):
    """(A, b, lo, hi, bounded mask) of one case, seeded by the case."""
    rng = np.random.default_rng(1000 * D + 10 * SCALES.index(scale) + KINDS.index(kind))
    nb = int(round(0.68 * D))
    m = int(0.9 * D) + 4  # fewer rows than unknowns for the larger D: J'J alone is singular, the damping makes A SPD
    J = rng.normal(size=(m, D)) * scale
    e = rng.normal(size=m) * 0.05 * max(scale, 1.0)  # J * 1e-3 with a 1e-3 residual would be all damping
    A = J.T @ J + (1e-3 + e @ e) * np.eye(D)
    b = J.T @ e
    bounded = np.zeros(D, bool)
    bounded[D - nb:] = True
    xu = -np.linalg.solve(A, b)
    mag = np.abs(xu[bounded])
    lim = {"none": 2.0 * mag.max(), "half": float(np.median(mag)), "all": 1e-4, "zero": 0.0,
           "degenerate_free": 2.0 * mag.max(), "degenerate_mixed": float(np.median(mag))}[kind]
    lo, hi = np.full(D, -np.inf), np.full(D, np.inf)
    lo[bounded], hi[bounded] = -lim, lim
    if kind == "degenerate_free":
        # the unconstrained optimum of the largest bounded unknown sits exactly on its upper / lower bound
        k = int(np.nonzero(bounded)[0][np.argmax(mag)])
        (hi if xu[k] > 0 else lo)[k] = xu[k]
    elif kind == "degenerate_mixed":
        # with about half of the bounds active, move one interior unknown's bound onto its optimal value
        x = q.reference_box_qp(A, b, lo, hi)
        inner = np.nonzero(bounded & (np.abs(x) < 0.5 * lim))[0]
        k = int(inner[np.argmax(np.abs(x[inner]))])
        (hi if x[k] > 0 else lo)[k] = x[k]
    return A, b, lo, hi, bounded


@pytest.fixture(scope="module")
def solved():
    cache = {}

    def get(D, scale, kind):
        if (D, scale, kind) not in cache:
            from oracle.smpl_oracle import solve_box_qp
            A, b, lo, hi, bounded = make_problem(D, scale, kind)
            cache[(D, scale, kind)] = (A, b, lo, hi, bounded, q.reference_box_qp(A, b, lo, hi), solve_box_qp(A, b, lo, hi))
        return cache[(D, scale, kind)]
    return get


@pytest.mark.parametrize("D,scale,kind", CASES, ids=["D%d-J%g-%s" % c for c in CASES])
def test_certificate_accepts_bvls_and_active_set(solved, D, scale, kind):
    A, b, lo, hi, bounded, x_ref, x_as = solved(D, scale, kind)
    for name, x in (("bvls", x_ref), ("solve_box_qp", x_as)):
        ok, rep = q.kkt_certificate(A, b, x, lo, hi)
        assert ok, (name, rep)
    active = np.abs(q.active_set(x_as, lo, hi)).sum()
    pinned = int((lo == hi).sum())
    if kind in ("none", "degenerate_free"):
        assert active <= 1 and pinned == 0
    elif kind in ("half", "degenerate_mixed"):
        assert 0.1 * bounded.sum() <= active <= 0.9 * bounded.sum()
    elif kind == "all":
        assert active >= 0.5 * bounded.sum()
    else:
        assert active == 0 and pinned == bounded.sum() and (x_as[bounded] == 0).all()
    # the two solvers reach the same optimum (A can be ill-conditioned, so the objective, not x, is compared)
    f_ref, f_as = q.objective(A, b, x_ref), q.objective(A, b, x_as)
    tol = q.objective_gap_tol(A, b, x_as)
    assert abs(f_as - f_ref) <= tol, (f_as, f_ref, tol)


def _weakest_active(A, b, x, lo, hi):
    """The active unknown with the smallest multiplier that is still clearly positive (> 1e-8 s): the bound an early
    stop or a wrong active set gets wrong first."""
    lam = q.multipliers(A, b, x, lo, hi) / q.problem_scale(A, b, x)
    cand = np.nonzero(lam > 1e-8)[0]
    assert cand.size, "no clearly active bound"
    return int(cand[np.argmin(lam[cand])])


REJECT = [(d, s, k) for d in SIZES for s in SCALES for k in ("half", "all", "degenerate_mixed")]


@pytest.mark.parametrize("D,scale,kind", REJECT, ids=["D%d-J%g-%s" % c for c in REJECT])
def test_certificate_rejects_subtly_wrong_steps(solved, D, scale, kind):
    A, b, lo, hi, bounded, x_ref, x_as = solved(D, scale, kind)
    k = _weakest_active(A, b, x_as, lo, hi)
    # an active unknown 1e-6 of its limit inside the box (a solve that stopped short of the bound)
    moved = x_as.copy()
    moved[k] -= 1e-6 * moved[k]
    ok, rep = q.kkt_certificate(A, b, moved, lo, hi)
    assert not ok and "interior" in rep["worst"], rep
    # the same unknown at its other bound (a wrong active set)
    flipped = x_as.copy()
    flipped[k] = lo[k] if x_as[k] >= hi[k] else hi[k]
    assert not q.kkt_certificate(A, b, flipped, lo, hi)[0]
    # the plain Cholesky step clipped to the box
    clipped = np.clip(-np.linalg.solve(A, b), lo, hi)
    assert not q.kkt_certificate(A, b, clipped, lo, hi)[0]


@pytest.mark.parametrize("D", SIZES)
def test_certificate_rejects_clipped_step_with_zero_limits(solved, D):
    """With every bounded unknown pinned at 0, the unconstrained step with those entries zeroed is not the solution
    (the unbounded unknowns must re-solve their own block)."""
    A, b, lo, hi, bounded, _, x_as = solved(D, 1.0, "zero")
    assert q.kkt_certificate(A, b, x_as, lo, hi)[0]
    assert not q.kkt_certificate(A, b, np.clip(-np.linalg.solve(A, b), lo, hi), lo, hi)[0]
    free = ~bounded
    x_free = np.zeros(D)
    x_free[free] = -np.linalg.solve(A[np.ix_(free, free)], b[free])
    assert np.abs(x_free - x_as).max() <= 1e-9 * np.abs(x_free).max()


def test_ik_bounds_layout():
    n, th = 3, 75
    lo, hi = q.ik_bounds(dict(enable_phi=1, phi_limit=0.04, optimize_beta=1, delta_beta_limit=0.01), n, th + 6 + 10, th)
    assert np.isinf(lo[:th]).all() and np.isinf(hi[:th]).all()
    assert (hi[th:th + 6] == float(np.float32(0.04))).all() and (lo[th:th + 6] == -float(np.float32(0.04))).all()
    assert (hi[th + 6:] == float(np.float32(0.01))).all()
    # phi off (or a zero limit): the phi entries of delta are exactly 0
    lo, hi = q.ik_bounds(dict(enable_phi=0, phi_limit=0.04), n, th + 6, th)
    assert (lo[th:] == 0).all() and (hi[th:] == 0).all()
    lo, hi = q.ik_bounds(dict(enable_phi=1, phi_limit=0.0), n, th + 6, th)
    assert (lo[th:] == 0).all() and (hi[th:] == 0).all()
    # no QP: existing phi / beta columns are unbounded
    lo, hi = q.ik_bounds(dict(enable_qp=0, enable_phi=1, phi_limit=0.04, optimize_beta=1), n, th + 16, th)
    assert np.isinf(lo).all() and np.isinf(hi).all()
    # a pinned unknown has no sign condition, an unknown outside its box fails whatever its gradient
    A, b = np.eye(2), np.array([1.0, -1.0])
    assert q.kkt_certificate(A, b, np.zeros(2), np.zeros(2), np.zeros(2))[0]
    ok, rep = q.kkt_certificate(A, b, np.array([0.0, 2e-12]), np.full(2, -1e-12), np.full(2, 1e-12))
    assert not ok and "outside" in rep["worst"]
