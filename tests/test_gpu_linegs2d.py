"""Zebra line Gauss-Seidel (SMOOTHER_LINE_GS) on the device against its CPU oracle
(tests/oracle_linegs2d.py): per-level iterates of whole V-cycles, fast arithmetic, the stand-alone
smoother, device and host setup, iteration counts, PCG, the rejections, and anisotropic 4097^2."""
import importlib

import numpy as np
import pytest
import scipy.sparse as sp

import oracle as O
import oracle_linegs2d as OL

amg = importlib.import_module("algebraic-multigrid_b200")
pytestmark = pytest.mark.gpu

LINES = {"x": amg.LINES_X, "y": amg.LINES_Y, "alt": amg.LINES_ALTERNATING}


def n_levels(m, min_lines=4):
    L = 1
    while m // 2 >= min_lines:
        m //= 2
        L += 1
    return L


def pair(m, lines="x", eps=1.0, L=None, every=10, n_iters=100, tol=1e-9, iters=1, **kw):
    L = L or n_levels(m)
    A, b = amg.Grid.laplacian(m, eps), amg.Grid.rhs(m)
    mg = amg.Multigrid(amg.BilinearInterpolator2D(L), amg.LineGaussSeidel(iters, LINES[lines]), A, b, L, tol,
                       every, n_iters, **kw)
    mo = OL.Multigrid(O.laplacian(m, eps), b, L, tol, every, n_iters, OL.SMOOTHER_LINE_GS, iters,
                      lines=LINES[lines])
    return mg, mo


def same_bytes(a, b):
    return np.asarray(a).tobytes() == np.asarray(b).tobytes()


@pytest.mark.parametrize("m", [35, 64, 65, 100, 257])
@pytest.mark.parametrize("eps", [1.0, 1e-3, 1e3])
@pytest.mark.parametrize("lines", ["x", "y", "alt"])
def test_vcycles_bit_exact_per_level(m, eps, lines):
    mg, mo = pair(m, lines, eps)
    for _ in range(2):
        mg.vcycle()
        mo.vcycle()
        for l in range(mg.n_levels):
            assert same_bytes(mg.get_rhs(l), mo.f(l)), ("f", l)
            assert same_bytes(mg.get_soln(l), mo.u(l)), ("u", l)


@pytest.mark.parametrize("m", [64, 65, 257])
@pytest.mark.parametrize("lines", ["x", "alt"])
def test_fast_arithmetic_within_1e12(m, lines):
    mg, mo = pair(m, lines, 1e-3, arith=amg.ARITH_FAST)
    for _ in range(3):
        mg.vcycle()
        mo.vcycle()
    u, uo = mg.get_soln(0), mo.u(0)
    assert np.linalg.norm(u - uo) / np.linalg.norm(uo) <= 1e-12


@pytest.mark.parametrize("m", [35, 64, 100])
@pytest.mark.parametrize("lines", ["x", "y", "alt"])
def test_standalone_smoother_bit_exact(m, lines):
    A = amg.Grid.laplacian(m, 1e-2)
    rng = np.random.default_rng(m)
    b, u = rng.standard_normal(m * m), rng.standard_normal(m * m)
    want = u.copy()
    OL.LineSmoother(O.laplacian(m, 1e-2), LINES[lines]).smooth(b, want, 2)
    amg.LineGaussSeidel(2, LINES[lines]).smooth(A, u, b)
    assert same_bytes(u, want)


@pytest.mark.parametrize("lines", ["x", "alt"])
def test_device_and_host_setup_agree(monkeypatch, lines):
    m = 129
    mg, _ = pair(m, lines, 1e-3)
    monkeypatch.setenv("AMGB_HOST_SETUP", "1")
    mh, _ = pair(m, lines, 1e-3)
    for _ in range(2):
        mg.vcycle()
        mh.vcycle()
    for l in range(mg.n_levels):
        assert same_bytes(mg.get_soln(l), mh.get_soln(l)), l


@pytest.mark.parametrize("m,eps,lines", [(65, 1e-3, "x"), (100, 1.0, "alt"), (65, 1e3, "y")])
def test_iteration_counts_equal_oracle(m, eps, lines):
    b = amg.Grid.rhs(m)
    tol = (1e-8 * np.linalg.norm(b)) ** 2  # rss criterion of solve()
    mg, mo = pair(m, lines, eps, every=1, n_iters=50, tol=tol)
    mg.solve()
    mo.solve()
    assert mg.iters_done == mo.iters_done and mg.iters_done < 50
    mg, mo = pair(m, lines, eps, every=1, n_iters=50)
    mg.solve_relative(1e-8)
    mo.solve_relative(1e-8)
    assert mg.iters_done == mo.iters_done and mg.iters_done < 50


def test_pcg_with_line_gs_cycle():
    m = 129
    mg, _ = pair(m, "x", 1e-3, n_iters=100)
    mg.solve_pcg(1e-8, 100)
    assert mg.last_error <= 1e-8, (mg.iters_done, mg.last_error)


def test_smooth_level_and_timing_hooks():
    m = 129
    mg, mo = pair(m, "alt", 1e-3)
    mg.vcycle()
    mo.vcycle()
    for l in range(mg.n_levels - 1):
        mg.smooth_level(l)
        mo.smooth(l)
        assert same_bytes(mg.get_soln(l), mo.u(l)), l
    for kind in (0, 12, 13):
        assert mg.time_kernel(0, kind, 1, 2) > 0.0
    assert mg.launches_per_vcycle() > 0
    mj = amg.Multigrid(amg.BilinearInterpolator2D(3), amg.DampedJacobi(), amg.Grid.laplacian(65), amg.Grid.rhs(65), 3)
    with pytest.raises(amg.AmgbError):
        mj.time_kernel(0, 12, 1, 1)


def test_rejections():
    m = 33
    A, b = amg.Grid.laplacian(m, 1e-3), amg.Grid.rhs(m)
    # the linear transfer
    with pytest.raises(ValueError, match="bilinear"):
        amg.Multigrid(amg.LinearInterpolator(3), amg.LineGaussSeidel(), A, b, 3)
    # a sharded create, one-rank communicator
    comm = amg.Comm(0, 1, lambda raw: raw)
    with pytest.raises(ValueError, match="single-GPU"):
        amg.Multigrid(amg.BilinearInterpolator2D(3), amg.LineGaussSeidel(), A, b, 3, comm=comm)
    # an unknown `lines` value (past the Python check)
    s = amg.LineGaussSeidel()
    s.lines = 7
    with pytest.raises(ValueError, match="line direction"):
        amg.Multigrid(amg.BilinearInterpolator2D(3), s, A, b, 3)
    with pytest.raises(ValueError):
        s.smooth(A, np.zeros(m * m), b)
    # +-2 coupling along a line: level 0 is not a 3 x 3 grid stencil
    M = sp.csc_matrix(A.to_scipy() + sp.kron(sp.identity(m), sp.diags([-0.1, -0.1], [-2, 2], shape=(m, m))))
    M.sort_indices()
    W = amg.CscMatrix(m * m, m * m, M.indptr, M.indices, M.data)
    with pytest.raises(ValueError, match="level 0"):
        amg.Multigrid(amg.BilinearInterpolator2D(3), amg.LineGaussSeidel(), W, b, 3)
    with pytest.raises(ValueError, match="grid operator"):
        amg.LineGaussSeidel().smooth(W, np.zeros(m * m), b)
    # a zero pivot: row k of the X-line solve has a_kk = a_k,k-1 = 0 (den_k = 0)
    k = 5 * m + 7
    Z = sp.lil_matrix(A.to_scipy())
    Z[k, k] = 0.0
    Z[k, k - 1] = 0.0
    Z = sp.csc_matrix(Z)
    Z.eliminate_zeros()
    Z.sort_indices()
    Zm = amg.CscMatrix(m * m, m * m, Z.indptr, Z.indices, Z.data)
    with pytest.raises(ValueError, match="level 0.*row %d" % k):
        amg.Multigrid(amg.BilinearInterpolator2D(3), amg.LineGaussSeidel(), Zm, b, 3)
    with pytest.raises(ValueError, match="row %d" % k):
        amg.LineGaussSeidel().smooth(Zm, np.zeros(m * m), b)


def host_rel_residual(m, eps, u, b):
    A = amg.Grid.laplacian(m, eps).to_scipy()
    return np.linalg.norm(b - A @ u) / np.linalg.norm(b)


@pytest.mark.parametrize("eps,lines", [(1e-3, "x"), (1.0, "alt")])
def test_4097_reaches_1e8_within_10_cycles(eps, lines):
    m = 4097
    L = n_levels(m, 8)
    A, b = amg.Grid.laplacian(m, eps), amg.Grid.rhs(m)
    mg = amg.Multigrid(amg.BilinearInterpolator2D(L), amg.LineGaussSeidel(1, LINES[lines]), A, b, L, 1e-9, 1, 10,
                       arith=amg.ARITH_FAST)
    mg.solve_relative(1e-8)
    assert mg.iters_done <= 10 and mg.last_error <= 1e-8, (mg.iters_done, mg.last_error)
    assert host_rel_residual(m, eps, mg.get_soln(0), b) <= 1e-8


def test_4097_aniso_damped_jacobi_does_not_reach_1e8_in_30_cycles():
    m = 4097
    L = n_levels(m, 8)
    A, b = amg.Grid.laplacian(m, 1e-3), amg.Grid.rhs(m)
    mg = amg.Multigrid(amg.BilinearInterpolator2D(L), amg.DampedJacobi(2.0 / 3.0, 2), A, b, L, 1e-9, 1, 30,
                       arith=amg.ARITH_FAST)
    mg.solve_relative(1e-8)
    assert host_rel_residual(m, 1e-3, mg.get_soln(0), b) > 1e-8
