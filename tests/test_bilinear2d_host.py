"""CPU checks of the bilinear 2-D transfer (TRANSFER_BILINEAR_2D): the operators the C ABI builds,
the coarse-size rule, the row-wise device Galerkin product (galerkin_dia2d.cuh compiled on the host)
against the oracle's Eigen-order product, and the convergence the 2-D hierarchy buys."""
import ctypes as C
import importlib
import os
import subprocess
import tempfile

import numpy as np
import pytest
import scipy.sparse as sp

import oracle as O
import oracle_bilinear2d as O2

amg = importlib.import_module("algebraic-multigrid_b200")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIZES = [2, 3, 35, 36, 64, 65, 100]


@pytest.mark.parametrize("m_h", SIZES)
def test_operators_are_kron_of_the_linear_pattern(m_h):
    m_H = amg.lib().amgb_bilinear_coarse_lines(m_h)
    bi = amg.BilinearInterpolator2D(2)
    bi.make_operators(m_h * m_h, m_H * m_H, 0)
    P, R = bi.get_P(0), bi.get_R(0)
    P1 = O.make_P(m_h, m_H).to_scipy()
    want = sp.csc_matrix(sp.kron(P1, P1))
    want.sort_indices()
    np.testing.assert_array_equal(P.colptr, want.indptr)
    np.testing.assert_array_equal(P.rowidx, want.indices)
    assert P.val.tobytes() == want.data.tobytes()
    wantR = sp.csc_matrix(want.T)
    wantR.sort_indices()
    np.testing.assert_array_equal(R.colptr, wantR.indptr)
    np.testing.assert_array_equal(R.rowidx, wantR.indices)
    assert R.val.tobytes() == wantR.data.tobytes()
    # and the oracle's P is the same matrix
    c, r, v = O2.make_P2d(m_h, m_H).arrays()
    np.testing.assert_array_equal(P.colptr, c)
    np.testing.assert_array_equal(P.rowidx, r)
    assert P.val.tobytes() == v.tobytes()


def test_coarse_rule_is_half_the_lines():
    for m in range(0, 300):
        assert amg.lib().amgb_bilinear_coarse_lines(m) == m // 2 == O2.coarse_lines(m)


def test_make_operators_rejects_sizes_off_the_rule():
    bi = amg.BilinearInterpolator2D(2)
    with pytest.raises(ValueError):
        bi.make_operators(35 * 35, 18 * 18, 0)   # 35 // 2 = 17
    with pytest.raises(ValueError):
        bi.make_operators(35 * 35 + 1, 17 * 17, 0)


# ---- galerkin_dia2d.cuh on the host -------------------------------------------------------------

def _gal2d_lib():
    src = os.path.join(ROOT, "tests", "cpp", "galerkin_dia2d_host.cpp")
    out = os.path.join(tempfile.mkdtemp(prefix="amgb_gal2d_"), "libgalerkin_dia2d_host.so")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-Wall",
                           "-x", "c++", src, "-o", out])
    L = C.CDLL(out)
    pd = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")
    pi = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
    L.gal2d_host_coarse.restype = None
    L.gal2d_host_coarse.argtypes = [C.c_int, C.c_int, pi, C.c_int, pd, C.c_int, pi, C.POINTER(C.c_int), C.c_int, pd]
    return L


@pytest.fixture(scope="module")
def gal2d():
    return _gal2d_lib()


def rows_dia(A):
    """DIA of the ROWS of A: val[d, i] = A(i, i + off[d]), explicit zeros dropped."""
    colptr, rowidx, val = A.arrays()
    n = A.cols
    cols = np.repeat(np.arange(n, dtype=np.int64), np.diff(colptr))
    keep = val != 0.0
    rows = rowidx.astype(np.int64)[keep]
    offs = cols[keep] - rows
    uniq = np.unique(offs)
    ld = (n + 31) // 32 * 32
    D = np.zeros((len(uniq), ld))
    D[np.searchsorted(uniq, offs), rows] = val[keep]
    return uniq.astype(np.int32), ld, D


def nine_point_unsymmetric(m, seed=7):
    """An unsymmetric 9-point grid operator with irregular values (oracle CSC)."""
    rng = np.random.default_rng(seed)
    rows, cols, vals = [], [], []
    for y in range(m):
        for x in range(m):
            k = y * m + x
            for dy in (-1, 0, 1):
                for dx in (-1, 0, 1):
                    yy, xx = y + dy, x + dx
                    if 0 <= yy < m and 0 <= xx < m:
                        rows.append(yy * m + xx)
                        cols.append(k)
                        vals.append(8.0 + rng.random() if (dy, dx) == (0, 0) else -rng.random())
    M = sp.csc_matrix((vals, (rows, cols)), shape=(m * m, m * m))
    M.sort_indices()
    return O.Csc.from_arrays(m * m, m * m, M.indptr, M.indices, M.data)


def _check_level(L, A, m_h):
    m_H = m_h // 2
    P = O2.make_P2d(m_h, m_H)
    want = O.galerkin(P.transpose(), A, P)
    off_f, ld_f, D_f = rows_dia(A)
    n_c = m_H * m_H
    ld_c = max(32, (n_c + 31) // 32 * 32)
    off_c = np.zeros(9, np.int32)
    nd_c = C.c_int(0)
    val_c = np.zeros(9 * ld_c)
    L.gal2d_host_coarse(m_h, len(off_f), off_f, ld_f, D_f.reshape(-1).copy(), m_H, off_c, C.byref(nd_c), ld_c, val_c)
    got = {int(off_c[c]): val_c[c * ld_c:c * ld_c + n_c] for c in range(nd_c.value)}
    want_off, _, want_D = rows_dia(want)
    for d, o in enumerate(want_off):
        assert int(o) in got, (m_h, o)
        assert got[int(o)].tobytes() == want_D[d, :n_c].tobytes(), (m_h, int(o))
    for o, v in got.items():
        if o not in set(int(x) for x in want_off):
            assert not v.any(), (m_h, o)
    return want


@pytest.mark.parametrize("m", SIZES)
@pytest.mark.parametrize("eps", [1.0, 1e-3])
def test_rowwise_galerkin_2d_matches_eigen_order_product(gal2d, m, eps):
    A, m_h = O.laplacian(m, eps), m
    while m_h // 2 >= 1:  # every level of the hierarchy
        A = _check_level(gal2d, A, m_h)
        m_h //= 2


@pytest.mark.parametrize("m", [3, 35, 36, 64])
def test_rowwise_galerkin_2d_unsymmetric_nine_point(gal2d, m):
    A, m_h = nine_point_unsymmetric(m), m
    while m_h // 2 >= 1:
        A = _check_level(gal2d, A, m_h)
        m_h //= 2


# ---- convergence of the 2-D hierarchy (oracle) ----------------------------------------------------

def levels_2d(m):
    """Coarsen while the coarse grid keeps at least 15 lines (exact solve below)."""
    L = 1
    while m // 2 >= 15:
        m //= 2
        L += 1
    return L


def levels_1d(n):
    L = 1
    while n > 20:
        n = O.n_H_from_n_h(n)
        L += 1
    return L


@pytest.mark.parametrize("m", [63, 100, 129])
@pytest.mark.parametrize("smoother,iters,cap", [(O.SMOOTHER_JACOBI, 2, 12), (O.SMOOTHER_GS, 1, 8)])
def test_2d_hierarchy_converges_where_1d_does_not(m, smoother, iters, cap):
    A, b = O.laplacian(m), O.rhs(m)
    mg = O2.Multigrid(A, b, levels_2d(m), 1e-9, 1, cap, smoother, iters, 2.0 / 3.0)
    mg.solve_relative(1e-8)
    r = O.residual(A, mg.u(0), b)
    assert mg.last_error <= 1e-8 and mg.iters_done <= cap, (mg.iters_done, mg.last_error)
    assert np.linalg.norm(r) / np.linalg.norm(b) <= 1e-8
    m1 = O.Multigrid(A, b, levels_1d(m * m), 1e-9, 1, cap, smoother, iters, 2.0 / 3.0)
    for _ in range(cap):
        m1.vcycle()
    rel1 = np.linalg.norm(O.residual(A, m1.u(0), b)) / np.linalg.norm(b)
    assert rel1 > 1e-8, rel1
