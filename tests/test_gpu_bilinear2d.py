"""The bilinear 2-D transfer (TRANSFER_BILINEAR_2D) on the device against its CPU oracle
(tests/oracle_bilinear2d.py): level operators, per-level iterates of whole V-cycles, the stand-alone
transfers, iteration counts, and the grid-size independent convergence at 4097^2."""
import importlib

import numpy as np
import pytest
import scipy.sparse as sp

import oracle as O
import oracle_bilinear2d as O2

amg = importlib.import_module("algebraic-multigrid_b200")
pytestmark = pytest.mark.gpu

SMOOTHERS = {
    "jacobi": (lambda: amg.DampedJacobi(2.0 / 3.0, 2), O.SMOOTHER_JACOBI, 2),
    "color_gs": (lambda: amg.MulticolorGaussSeidel(1), O.SMOOTHER_COLOR_GS, 1),
    "gs_auto": (lambda: amg.SparseGaussSeidel(mode=amg.GS_AUTO), O.SMOOTHER_GS, 1),
}


def n_levels(m, min_lines=4):
    L = 1
    while m // 2 >= min_lines:
        m //= 2
        L += 1
    return L


def pair(m, smoother, L=None, eps=1.0, every=10, n_iters=100, tol=1e-9, **kw):
    make, kind, iters = SMOOTHERS[smoother]
    L = L or n_levels(m)
    A, b = amg.Grid.laplacian(m, eps), amg.Grid.rhs(m)
    mg = amg.Multigrid(amg.BilinearInterpolator2D(L), make(), A, b, L, tol, every, n_iters, **kw)
    mo = O2.Multigrid(O.laplacian(m, eps), b, L, tol, every, n_iters, kind, iters, 2.0 / 3.0)
    return mg, mo, A, b


def same_bytes(a, b):
    return np.asarray(a).tobytes() == np.asarray(b).tobytes()


@pytest.mark.parametrize("m", [35, 64, 65, 100])
@pytest.mark.parametrize("smoother", ["jacobi", "gs_auto"])
def test_level_operators_match_oracle(m, smoother):
    mg, mo, _, _ = pair(m, smoother)
    assert mg.transfer() == amg.TRANSFER_BILINEAR_2D
    for l in range(mg.n_levels):
        assert mg.get_n_dofs(l) == mo.n_dofs(l) == mo.m[l] ** 2
        M = mg.get_coefficient_matrix(l)
        c, r, v = mo.A(l).arrays()
        np.testing.assert_array_equal(M.colptr, c)
        np.testing.assert_array_equal(M.rowidx, r)
        assert same_bytes(M.val, v), l
    if smoother == "jacobi":  # device DIA levels (device setup) against the host product
        for l in range(mg.n_levels - 1):
            _, bad = mg.galerkin_device(l)
            assert bad == 0, l


@pytest.mark.parametrize("m", [35, 64, 65, 100, 257])
@pytest.mark.parametrize("smoother", ["jacobi", "color_gs", "gs_auto"])
@pytest.mark.parametrize("eps", [1.0, 1e-3])
def test_one_vcycle_bit_exact_per_level(m, smoother, eps):
    mg, mo, _, _ = pair(m, smoother, eps=eps)
    for _ in range(2):
        mg.vcycle()
        mo.vcycle()
        for l in range(mg.n_levels):
            assert same_bytes(mg.get_rhs(l), mo.f(l)), ("f", l)
            assert same_bytes(mg.get_soln(l), mo.u(l)), ("u", l)


@pytest.mark.parametrize("m", [35, 64])
def test_operator_beyond_3x3_stencil_uses_host_product(m):
    """A damped-Jacobi 2-D hierarchy whose operator couples points two apart along a line is not a
    3 x 3 grid stencil: the device setup leaves it to the host product, which must match the oracle."""
    L = n_levels(m)
    A5 = amg.Grid.laplacian(m).to_scipy()
    T = sp.diags([np.full(m - 2, 0.05), np.full(m - 2, 0.05)], [-2, 2]) * (m + 1) ** 2
    M = sp.csc_matrix(A5 + sp.kron(sp.identity(m), T))
    M.sort_indices()
    A = amg.CscMatrix(m * m, m * m, M.indptr, M.indices, M.data)
    b = amg.Grid.rhs(m)
    mg = amg.Multigrid(amg.BilinearInterpolator2D(L), amg.DampedJacobi(2.0 / 3.0, 2), A, b, L, 1e-9, 10, 100)
    mo = O2.Multigrid(O.Csc.from_arrays(m * m, m * m, M.indptr, M.indices, M.data), b, L, 1e-9, 10, 100,
                      O.SMOOTHER_JACOBI, 2, 2.0 / 3.0)
    for l in range(L):
        Mg = mg.get_coefficient_matrix(l)
        c, r, v = mo.A(l).arrays()
        np.testing.assert_array_equal(Mg.colptr, c)
        np.testing.assert_array_equal(Mg.rowidx, r)
        assert same_bytes(Mg.val, v), l
    mg.vcycle()
    mo.vcycle()
    for l in range(L):
        assert same_bytes(mg.get_soln(l), mo.u(l)), l


@pytest.mark.parametrize("m", [64, 65, 257])
def test_fast_arithmetic_within_1e12(m):
    mg, mo, _, _ = pair(m, "jacobi", arith=amg.ARITH_FAST)
    for _ in range(3):
        mg.vcycle()
        mo.vcycle()
    u, uo = mg.get_soln(0), mo.u(0)
    assert np.linalg.norm(u - uo) / np.linalg.norm(uo) <= 1e-12


@pytest.mark.parametrize("m", [35, 64, 65, 100])
def test_standalone_transfers_bit_exact(m):
    mg, mo, _, _ = pair(m, "jacobi")
    rng = np.random.default_rng(m)
    for l in range(mg.n_levels - 1):
        nf, nc = mo.n_dofs(l), mo.n_dofs(l + 1)
        r, e, u = rng.standard_normal(nf), rng.standard_normal(nc), rng.standard_normal(nf)
        assert same_bytes(mg.restrict(l, r), O.spmv(mo.R(l), r)), l
        assert same_bytes(mg.prolong_add(l, e, u), u + O.spmv(mo.P(l), e)), l
        f = rng.standard_normal(nf)
        mg.set_soln(l, u)
        mg.set_rhs(l, f)
        mg.set_soln(l + 1, e)
        mg.residual_restrict_level(l)
        assert same_bytes(mg.get_rhs(l + 1), O.spmv(mo.R(l), O.residual(mo.A(l), u, f))), l
        assert not mg.get_soln(l + 1).any()


@pytest.mark.parametrize("m", [35, 64, 65, 257])
def test_wavefront_gauss_seidel_on_every_level(m):
    mg, mo, _, _ = pair(m, "gs_auto", L=n_levels(m, 2))
    for l in range(mg.n_levels):
        if mo.m[l] >= 3:
            assert mg.gs_kernel(l) == amg.GS_KERNEL_WAVE, l


@pytest.mark.parametrize("m", [65, 100])
@pytest.mark.parametrize("smoother", ["jacobi", "gs_auto"])
def test_iteration_counts_equal_oracle(m, smoother):
    b = amg.Grid.rhs(m)
    tol = (1e-8 * np.linalg.norm(b)) ** 2  # rss criterion of solve()
    mg, mo, _, _ = pair(m, smoother, every=1, n_iters=50, tol=tol)
    mg.solve()
    mo.solve()
    assert mg.iters_done == mo.iters_done and mg.iters_done < 50
    mg, mo, _, _ = pair(m, smoother, every=1, n_iters=50)
    mg.solve_relative(1e-8)
    mo.solve_relative(1e-8)
    assert mg.iters_done == mo.iters_done and mg.iters_done < 50


def test_pcg_takes_fewer_iterations_with_2d_hierarchy():
    m = 129
    A, b = amg.Grid.laplacian(m), amg.Grid.rhs(m)
    its = {}
    for name, interp, L in (("linear", amg.LinearInterpolator, 8), ("bilinear", amg.BilinearInterpolator2D, 6)):
        mg = amg.Multigrid(interp(L), amg.DampedJacobi(2.0 / 3.0, 2), A, b, L, 1e-9, 1, 1000)
        mg.solve_pcg(1e-8, 1000)
        assert mg.last_error <= 1e-8
        its[name] = mg.iters_done
    assert its["bilinear"] < its["linear"], its


def test_rejections_and_no_fused_paths():
    # non-square number of rows
    A1 = sp.diags([np.ones(29), -2 * np.ones(30), np.ones(29)], [-1, 0, 1], format="csc")
    A1.sort_indices()
    A = amg.CscMatrix(30, 30, A1.indptr, A1.indices, A1.data)
    with pytest.raises(ValueError):
        amg.Multigrid(amg.BilinearInterpolator2D(2), amg.DampedJacobi(), A, np.ones(30), 2)
    # a level that would be empty
    A, b = amg.Grid.laplacian(5), amg.Grid.rhs(5)
    with pytest.raises(ValueError):
        amg.Multigrid(amg.BilinearInterpolator2D(4), amg.DampedJacobi(), A, b, 4)  # 5 -> 2 -> 1 -> 0
    # sharded create, one-rank communicator
    comm = amg.Comm(0, 1, lambda raw: raw)
    A, b = amg.Grid.laplacian(64), amg.Grid.rhs(64)
    with pytest.raises(ValueError):
        amg.Multigrid(amg.BilinearInterpolator2D(3), amg.DampedJacobi(), A, b, 3, comm=comm)
    # fuse bits 1-7 do nothing on a 2-D hierarchy
    m = 257
    A, b = amg.Grid.laplacian(m), amg.Grid.rhs(m)
    mg = amg.Multigrid(amg.BilinearInterpolator2D(7), amg.DampedJacobi(2.0 / 3.0, 2), A, b, 7)
    assert all(not mg.fused_legs(l) for l in range(7))
    assert mg.tail_first() == -1
    assert mg.mid_range()[0] == -1
    lin = amg.Multigrid(amg.LinearInterpolator(7), amg.DampedJacobi(2.0 / 3.0, 2), A, b, 7)
    assert lin.transfer() == amg.TRANSFER_LINEAR


def host_rel_residual(m, u, b):
    A = amg.Grid.laplacian(m).to_scipy()
    return np.linalg.norm(b - A @ u) / np.linalg.norm(b)


@pytest.mark.parametrize("smoother,cap,kw", [("jacobi", 12, {"arith": amg.ARITH_FAST}), ("gs_auto", 8, {})])
def test_4097_converges_independently_of_grid_size(smoother, cap, kw):
    m = 4097
    make, _, _ = SMOOTHERS[smoother]
    L = n_levels(m, 8)
    A, b = amg.Grid.laplacian(m), amg.Grid.rhs(m)
    mg = amg.Multigrid(amg.BilinearInterpolator2D(L), make(), A, b, L, 1e-9, 1, 50, **kw)
    mg.solve_relative(1e-8)
    assert mg.iters_done <= cap, (mg.iters_done, mg.last_error)
    assert host_rel_residual(m, mg.get_soln(0), b) <= 1e-8
