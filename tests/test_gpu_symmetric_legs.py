"""Half-streaming register legs: on a level whose operator is bitwise symmetric the streaming legs
load only the centre and upper diagonals and take each lower coefficient from the row it couples
to.  The selection follows the operator, and the cycle stays bit-identical to the oracle."""
import importlib

import numpy as np
import pytest
import scipy.sparse as sp

import oracle as O

amg = importlib.import_module("algebraic-multigrid_b200")
pytestmark = pytest.mark.gpu

# grid size -> levels; odd n gives a seven-point level 1, even n a nine-point one
SIZES = [(35, 8), (64, 9), (65, 9), (100, 11), (129, 12), (257, 13), (1025, 14)]


def make_pair(A, Ao, b, L, nu):
    sm = amg.DampedJacobi(2.0 / 3.0, nu)
    mg = amg.Multigrid(amg.LinearInterpolator(L), sm, A, b, L, 1e-9, 1, 1)
    mo = O.Multigrid(Ao, b, L, 1e-9, 1, 1, O.SMOOTHER_JACOBI, nu, 2.0 / 3.0)
    return mg, mo


def streaming_levels(mg, L):
    return [l for l in range(L - 1) if mg.fused_legs(l) and mg.leg_plan(l)["smem_bytes"] == 0]


def check_selection(mg, L):
    """n_diagonals reports what a leg streams: half of the off-diagonals + the centre exactly on the
    streaming levels whose operator equals its transpose bit for bit, every diagonal elsewhere."""
    levels = streaming_levels(mg, L)
    assert levels
    n_half = 0
    for l in range(L):
        M = mg.get_coefficient_matrix(l)
        cols = np.repeat(np.arange(M.cols), np.diff(M.colptr))
        full = len(np.unique(M.rowidx - cols))
        S = sp.csc_matrix((M.val, M.rowidx, M.colptr), shape=(M.rows, M.cols))
        symmetric = (S != S.T).nnz == 0
        if l in levels and symmetric:
            assert full in (5, 7, 9), l
            assert mg.n_diagonals(l) == full // 2 + 1, l
            n_half += 1
        else:
            assert mg.n_diagonals(l) == full, l
    return levels, n_half


def check_cycles(mg, mo, L, cycles=3):
    for c in range(cycles):
        mg.vcycle(); mo.vcycle()
        for l in range(L):
            assert mg.get_soln(l).tobytes() == mo.u(l).tobytes(), (c, l)
            assert mg.get_rhs(l).tobytes() == mo.f(l).tobytes(), (c, l)


@pytest.mark.parametrize("nu", [1, 2])
@pytest.mark.parametrize("n,L", SIZES)
def test_half_streaming_isotropic(n, L, nu):
    """Every level of the isotropic Poisson hierarchy is bitwise symmetric: all streaming levels
    run half streaming, and the iterates after each of three cycles are the oracle's, bit for bit."""
    A, b, Ao = amg.Grid.laplacian(n), amg.Grid.rhs(n), O.laplacian(n)
    mg, mo = make_pair(A, Ao, b, L, nu)
    levels, n_half = check_selection(mg, L)
    assert n_half == len(levels)
    check_cycles(mg, mo, L)


@pytest.mark.parametrize("n,L", [(129, 12), (1025, 14)])
def test_half_streaming_anisotropic(n, L):
    """eps = 1e-3: levels 0-1 are bitwise symmetric, the Galerkin levels >= 2 are not (rounding), so
    one cycle runs both kinds of legs."""
    A, b, Ao = amg.Grid.laplacian(n, 1e-3), amg.Grid.rhs(n), O.laplacian(n, 1e-3)
    mg, mo = make_pair(A, Ao, b, L, 2)
    levels, n_half = check_selection(mg, L)
    assert 0 in levels and mg.n_diagonals(0) == 3
    assert any(l >= 2 and mg.n_diagonals(l) == 9 for l in levels)
    check_cycles(mg, mo, L)


def test_unsymmetric_operator_streams_every_diagonal():
    """A skewed operator (the one of test_asymmetric_operator_device_setup) keeps full streaming."""
    n, L = 65, 9
    A, b = amg.Grid.laplacian(n), amg.Grid.rhs(n)
    cols = np.repeat(np.arange(n * n), np.diff(A.colptr))
    A.val[A.rowidx < cols] *= 1.001
    Ao = O.Csc.from_arrays(A.rows, A.cols, A.colptr, A.rowidx, A.val)
    mg, mo = make_pair(A, Ao, b, L, 2)
    levels, n_half = check_selection(mg, L)
    assert n_half == 0 and mg.n_diagonals(0) == 5
    check_cycles(mg, mo, L, cycles=2)


@pytest.mark.parametrize("nu", [1, 2])
@pytest.mark.parametrize("n,L,eps", [(65, 9, 1.0), (100, 11, 1.0), (257, 13, 1.0), (129, 12, 1e-3)])
def test_half_streaming_short_chunks(n, L, eps, nu, monkeypatch):
    """Many chunks of one or two lines, so that chunk starts (and the extra operator line loaded
    before each chunk) fall on every line of the level, not only on line 0."""
    monkeypatch.setenv("AMGB_SLEG_MINLINES", "1" if nu == 1 else "2")
    monkeypatch.setenv("AMGB_SLEG_WARPS_PER_SM", "256")
    A, b, Ao = amg.Grid.laplacian(n, eps), amg.Grid.rhs(n), O.laplacian(n, eps)
    mg, mo = make_pair(A, Ao, b, L, nu)
    levels, n_half = check_selection(mg, L)
    assert n_half > 0
    check_cycles(mg, mo, L, cycles=2)
