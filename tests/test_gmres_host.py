"""tests/oracle_gmres.py, the specification of amgb_solve_gmres, without a GPU: right-preconditioned GMRES(m)
with one oracle V-cycle as the preconditioner converges where the stationary V-cycle diverges (upwind
convection-diffusion, unsymmetric Dirichlet elimination), in the step counts pinned here; the known limits are
pinned too; and the stopping rules (invariant subspace, ||b|| = 0, max_iters, restart) behave as specified."""
import functools

import numpy as np
import pytest
import scipy.sparse as sp

import oracle as O
import oracle_bilinear2d as B
import oracle_sa as S
import sa_matrices as G
from oracle_gmres import gmres

TOL = 1e-8
CAP = 25


def rhs(rows):
    return np.random.default_rng(rows).standard_normal(rows)


@functools.lru_cache(maxsize=None)
def matrix(name, n, pe=None):
    gen, theta, _ = G.FAMILIES[name]
    return (gen(n) if pe is None else G.convection(n, pe)), theta


def sa_run(name, n, gs=False, restart=30, max_iters=200, pe=None):
    A, theta = matrix(name, n, pe)
    b = rhs(A.rows)
    kind, iters = (O.SMOOTHER_GS, 1) if gs else (O.SMOOTHER_JACOBI, 2)
    mo = S.Multigrid(A, b, CAP, 1e-9, 1, 200, kind, iters, 2.0 / 3.0, theta)
    return gmres(A, b, lambda v: S.precondition(mo, v), TOL, restart, max_iters) + (A, b)


def check_converged(out):
    it, rel, x, hist, A, b = out
    assert rel <= TOL and len(hist) == it
    assert np.linalg.norm(b - A.to_scipy() @ x) / np.linalg.norm(b) == pytest.approx(rel, rel=1e-6)


@pytest.mark.parametrize("name,n,gs,steps", [
    ("conv", 129, False, 17), ("conv", 129, True, 20), ("conv", 257, False, 15), ("conv", 513, False, 19),
    ("dir", 65, False, 23), ("nine", 129, False, 12), ("neg", 129, False, 12), ("dirsym", 65, False, 10)])
def test_smoothed_aggregation_step_counts(name, n, gs, steps):
    out = sa_run(name, n, gs)
    assert out[0] == steps
    check_converged(out)


@pytest.mark.parametrize("m,steps", [(129, 10), (257, 9), (513, 9)])
def test_bilinear_convection_converges_where_the_stationary_cycle_diverges(m, steps):
    A, _ = matrix("conv", m)
    b = rhs(A.rows)
    L = int(np.log2(m + 1)) - 1
    mo = B.Multigrid(A, b, L, 1e-9, 1, 200, O.SMOOTHER_JACOBI, 2)
    out = gmres(A, b, lambda v: S.precondition(mo, v), TOL, 30, 200)
    assert out[0] == steps
    check_converged(out + (A, b))
    stationary = B.Multigrid(A, b, L, 1e-9, 1, 30, O.SMOOTHER_JACOBI, 2)
    stationary.solve_relative(TOL)
    assert not np.sqrt(stationary.rss()) / np.linalg.norm(b) < 1.0  # diverged (or overflowed to NaN)


@pytest.mark.parametrize("restart,steps", [(5, 19), (10, 17), (20, 15)])
def test_restart_sweep(restart, steps):
    out = sa_run("conv", 257, restart=restart)
    assert out[0] == steps
    check_converged(out)


def test_known_limits():
    """Pinned, not fixed: GMRES with these cycles does not reach 1e-8 within 200 steps."""
    it, rel, _, _, _, _ = sa_run("dir", 65, gs=True)
    assert it == 200 and 0.99 < rel < 1.0  # the Gauss-Seidel cycle on unsymmetric elimination stagnates
    it, rel, _, _, _, _ = sa_run("conv", 257, pe=1000.0)
    assert it == 200 and rel > TOL


def test_p1_finite_elements_stall_at_restart_30():
    it, rel, _, _, _, _ = sa_run("p1fe", 20000)
    assert it == 200 and rel > TOL


def test_three_distinct_eigenvalues_exhaust_the_krylov_space_in_three_steps():
    d = np.repeat([1.0, 2.0, 3.0], [5, 7, 9])
    A = sp.diags(d).tocsc()
    b = rhs(d.size)
    it, rel, x, hist = gmres(A, b, lambda v: v.copy(), 1e-14, 30, 100)
    assert it == 3 and len(hist) == 3
    assert hist[1] > 1e-3 and hist[2] < 1e-15  # the third step drops to round-off
    assert rel < 1e-14
    np.testing.assert_allclose(x, b / d, rtol=1e-13)


def test_exact_invariant_subspace_ends_the_cycle():
    """diag(3, 3, 1, 1), b = 1: the Arnoldi vectors are (1, 1, 1, 1) / 2 and (1, 1, -1, -1) / 2 exactly, so
    H(2, 1) is exactly 0 and, with rel_tol = 0, only that test ends the first cycle (without it, v_2 = w / 0).
    1/3 is inexact, so a second cycle of two steps removes the round-off left by the first."""
    A = sp.diags([3.0, 3.0, 1.0, 1.0]).tocsc()
    b = np.ones(4)
    it, rel, x, hist = gmres(A, b, lambda v: v.copy(), 0.0, 30, 100)
    assert it == 4 and hist[1] == 0.0 and 0.0 < hist[2] < 1e-15 and hist[3] == 0.0
    assert rel == 0.0 and np.allclose(x, [1 / 3, 1 / 3, 1.0, 1.0], rtol=1e-15)


def test_zero_rhs_and_zero_max_iters_return_at_once():
    A, theta = matrix("conv", 129)
    calls = []

    def prec(v):
        calls.append(1)
        return v.copy()

    it, rel, x, hist = gmres(A, np.zeros(A.rows), prec, TOL, 30, 100)
    assert (it, rel, hist, calls) == (0, 0.0, [], []) and not x.any()
    b = rhs(A.rows)
    x0 = np.full(A.rows, 0.5)
    it, rel, x, hist = gmres(A, b, prec, TOL, 30, 0, x0=x0)
    assert (it, hist, calls) == (0, [], [])
    assert x.tobytes() == x0.tobytes()
    assert rel == np.linalg.norm(b - A.to_scipy() @ x0) / np.linalg.norm(b)


def test_max_iters_is_a_hard_cap_inside_a_cycle():
    it, rel, _, hist, _, _ = sa_run("conv", 129, max_iters=7)
    assert it == 7 and len(hist) == 7 and rel > TOL
    # x was updated from the partial cycle: the true residual is near the last estimate
    assert rel == pytest.approx(hist[-1], rel=1e-3)


def test_restart_at_least_the_steps_needed_is_unrestarted_gmres():
    ref = sa_run("conv", 129, restart=1000)
    assert ref[0] == 17
    for restart in (17, 18, 40):
        out = sa_run("conv", 129, restart=restart)
        assert out[0] == ref[0] and out[2].tobytes() == ref[2].tobytes() and out[3] == ref[3]


def test_minimal_residual_property():
    """Within one cycle x_k minimises ||b - A M z|| over the Krylov space: compare with a dense least-squares
    solve on the same basis for a small unsymmetric matrix."""
    A, theta = matrix("conv", 33)
    b = rhs(A.rows)
    mo = S.Multigrid(A, b, CAP, 1e-9, 1, 200, O.SMOOTHER_JACOBI, 2, 2.0 / 3.0, theta)
    prec = lambda v: S.precondition(mo, v)  # noqa: E731
    As = A.to_scipy()
    for k in (1, 3, 6):
        it, rel, x, hist = gmres(A, b, prec, 0.0, k, k)
        K = [b / np.linalg.norm(b)]
        for _ in range(k - 1):
            K.append(As @ prec(K[-1]))
        Q, _ = np.linalg.qr(np.array(K).T)
        AMQ = np.column_stack([As @ prec(Q[:, i]) for i in range(k)])
        c, *_ = np.linalg.lstsq(AMQ, b, rcond=None)
        best = np.linalg.norm(b - AMQ @ c) / np.linalg.norm(b)
        assert it == k and rel == pytest.approx(best, rel=1e-6) and hist[-1] == pytest.approx(best, rel=1e-6)
