"""Smoothed-aggregation coarsening (TRANSFER_SMOOTHED_AGGREGATION) without a GPU: the C ABI's
amgb_sa_aggregate and the host setup of algebraic-multigrid_b200/csrc/host_setup.cpp against the numpy
oracle (tests/oracle_sa.py), the properties of the aggregates, the rejections, and the convergence of
the oracle's hierarchy where the 1-D transfer barely converges."""
import ctypes as C
import importlib
import os
import subprocess
import tempfile

import numpy as np
import pytest

import oracle as O
import oracle_sa as S

amg = importlib.import_module("algebraic-multigrid_b200")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "algebraic-multigrid_b200", "csrc")
_host = None


def host():
    """tests/cpp/sa_host.cpp + host_setup.cpp, built into a temporary directory."""
    global _host
    if _host is None:
        so = os.path.join(tempfile.mkdtemp(prefix="amgb_sa_host_"), "libsa_host.so")
        subprocess.check_call(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-Wall",
                               os.path.join(ROOT, "tests", "cpp", "sa_host.cpp"), os.path.join(CSRC, "host_setup.cpp"),
                               "-o", so])
        L = C.CDLL(so)
        pd = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")
        pi = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
        L.sa_host_build.argtypes = [C.c_int, pi, pi, pd, C.c_double, C.c_int]
        L.sa_host_error.restype = C.c_char_p
        L.sa_host_nnz.restype = C.c_longlong
        L.sa_host_copy.argtypes = [C.c_int, C.c_int, pi, pi, pd]
        _host = L
    return _host


def host_levels(A, n_levels, theta=0.08):
    """([A_l], [P_l]) as (colptr, rowidx, val) triples from the C++ host setup."""
    L = host()
    c, r, v = A.arrays()
    if L.sa_host_build(A.cols, c, r, v, theta, n_levels) != 0:
        raise ValueError(L.sa_host_error().decode())
    out = ([], [])
    for kind in (0, 1):
        for l in range(L.sa_host_n_levels() - kind):
            nnz = L.sa_host_nnz(kind, l)
            cp = np.empty(L.sa_host_cols(kind, l) + 1, np.int32)
            ri, va = np.empty(nnz, np.int32), np.empty(nnz)
            L.sa_host_copy(kind, l, cp, ri, va)
            out[kind].append((cp, ri, va))
    return out


def matrices():
    return {
        "iso65": O.laplacian(65),
        "eps1e-3_65": O.laplacian(65, 1e-3),
        "eps1e3_65": O.laplacian(65, 1e3),
        "rect70x31": S.rectangular_poisson(70, 31),
        "perm48": S.permuted_laplacian(48, seed=3)[0],
        "lognormal40": S.lognormal_diffusion(40, seed=5),
    }


MATS = matrices()


def as_amg(A):
    return amg.CscMatrix(A.rows, A.cols, *A.arrays())


def same_bytes(a, b):
    return np.asarray(a).tobytes() == np.asarray(b).tobytes()


@pytest.mark.parametrize("name", sorted(MATS))
def test_aggregate_matches_oracle_and_partitions_the_rows(name):
    A = MATS[name]
    agg, k = amg.sa_aggregate(as_amg(A))
    agg_o, k_o, _ = S.aggregate(A)
    assert k == k_o and 0 < k < A.rows
    np.testing.assert_array_equal(agg, agg_o)
    # every row in exactly one aggregate, every id used
    assert agg.min() == 0 and agg.max() == k - 1
    assert np.unique(agg).size == k


@pytest.mark.parametrize("name", sorted(MATS))
def test_pass1_aggregates_hold_their_roots_strong_neighbours(name):
    A = MATS[name]
    c, r, v = A.arrays()
    strong = S.strong(c, r, v, 0.08)
    agg, _, roots = S.aggregate(A)
    n1 = int((roots >= 0).sum())
    assert n1 > 0 and (roots[:n1] >= 0).all()
    for J, i in enumerate(roots[:n1]):
        nbrs = r[c[i]:c[i + 1]][strong[c[i]:c[i + 1]]]
        assert agg[i] == J and (agg[nbrs] == J).all()


def test_anisotropic_aggregates_stay_inside_one_x_line():
    m = 65
    agg, k = amg.sa_aggregate(as_amg(O.laplacian(m, 1e-3)))
    line = np.arange(m * m) // m
    for J in range(k):
        assert np.unique(line[agg == J]).size == 1, J


@pytest.mark.parametrize("name", sorted(MATS))
def test_host_prolongation_and_operators_bit_identical(name):
    A = MATS[name]
    As, Ps, _, _ = S.build(A, 10)
    hA, hP = host_levels(A, 10)
    assert len(hA) == len(As) >= 2 and len(hP) == len(Ps)
    for l, M in enumerate(As):
        c, r, v = M.arrays()
        np.testing.assert_array_equal(hA[l][0], c)
        np.testing.assert_array_equal(hA[l][1], r)
        assert same_bytes(hA[l][2], v), ("A", l)
    for l, M in enumerate(Ps):
        c, r, v = M.arrays()
        np.testing.assert_array_equal(hP[l][0], c)
        np.testing.assert_array_equal(hP[l][1], r)
        assert same_bytes(hP[l][2], v), ("P", l)


def test_stop_rule():
    A = O.laplacian(65)
    hA, _ = host_levels(A, 20)
    sizes = [c.shape[0] - 1 for c, _, _ in hA]
    assert sizes[-1] <= S.MAX_COARSE < sizes[-2]
    assert [M.rows for M in S.build(A, 20)[0]] == sizes
    assert len(host_levels(A, 2)[0]) == 2  # n_levels caps the hierarchy
    small = O.laplacian(14)  # 196 rows: nothing to coarsen
    assert len(host_levels(small, 5)[0]) == 1


def test_a_coarse_level_that_does_not_reduce_is_the_coarsest():
    # Poisson 129^2 with strength 0.15: level 5 (321 rows) has only weak couplings
    A = O.laplacian(129)
    hA, hP = host_levels(A, 25, 0.15)
    As, Ps, _, _ = S.build(A, 25, 0.15)
    assert [c.shape[0] - 1 for c, _, _ in hA] == [M.rows for M in As]
    assert len(As) == 6 and As[-1].rows > S.MAX_COARSE
    assert amg.sa_aggregate(as_amg(As[-1]), 0.15)[1] == As[-1].rows
    for l, M in enumerate(As):
        c, r, v = M.arrays()
        assert np.array_equal(hA[l][0], c) and np.array_equal(hA[l][1], r) and same_bytes(hA[l][2], v), l
    b = np.random.default_rng(2).standard_normal(A.rows)
    mg = S.Multigrid(A, b, 25, smoother=O.SMOOTHER_JACOBI, smoother_iters=2, theta=0.15)
    assert mg.n_levels == 6
    mg.solve_pcg(b, 1e-8, 100)
    assert mg.last_error <= 1e-8


def test_rejections():
    import scipy.sparse as sp
    # a diagonal matrix: every row is a singleton, the aggregation does not reduce level 0
    D = S._csc(sp.diags(np.arange(1.0, 301.0)))
    with pytest.raises(ValueError, match="level 0 does not reduce"):
        host_levels(D, 3)
    with pytest.raises(ValueError, match="does not reduce"):
        S.build(D, 3)
    # a zero diagonal: level and row are named
    L = O.laplacian(20).to_scipy().tolil()
    L[37, 37] = 0.0
    Z = S._csc(L)
    with pytest.raises(ValueError, match="level 0 has a zero diagonal at row 37"):
        host_levels(Z, 3)
    with pytest.raises(amg.InvalidArgument, match="row 37"):
        amg.sa_aggregate(as_amg(Z))
    with pytest.raises(ValueError, match="row 37"):
        S.aggregate(Z)
    # theta < 0 or NaN
    A = as_amg(O.laplacian(20))
    for theta in (-0.1, float("nan")):
        with pytest.raises(amg.InvalidArgument, match="strength"):
            amg.sa_aggregate(A, theta)
        with pytest.raises(ValueError, match="strength"):
            host_levels(O.laplacian(20), 3, theta)


# PCG to 1e-8 with the oracle's Jacobi 2+2 V-cycle; bounds fixed from the oracle's own counts
# (12, 14, 9, 8, 9, 10, 15, 17 when they were set) with a margin of two
CONVERGENCE = {
    "iso129": (lambda: O.laplacian(129), 14),
    "iso257": (lambda: O.laplacian(257), 16),
    "eps1e-3_129": (lambda: O.laplacian(129, 1e-3), 11),
    "eps1e-3_257": (lambda: O.laplacian(257, 1e-3), 10),
    "eps1e3_129": (lambda: O.laplacian(129, 1e3), 11),
    "rect300x120": (lambda: S.rectangular_poisson(300, 120), 12),
    "perm257": (lambda: S.permuted_laplacian(257)[0], 17),
    "lognormal129": (lambda: S.lognormal_diffusion(129), 19),
}


@pytest.mark.parametrize("name", sorted(CONVERGENCE))
def test_oracle_sa_pcg_converges_where_the_1d_transfer_does_not(name):
    make, bound = CONVERGENCE[name]
    A = make()
    b = np.random.default_rng(1).standard_normal(A.rows)
    mg = S.Multigrid(A, b, 25, smoother=O.SMOOTHER_JACOBI, smoother_iters=2)
    it = mg.solve_pcg(b, 1e-8, 100)
    assert mg.last_error <= 1e-8 and it <= bound, it
    if name.startswith("eps1e-3"):
        return  # the 1-D transfer semi-coarsens along the strong x-lines: it converges there too
    lin = O.Multigrid(A, b, 8, 1e-9, 10, 100, O.SMOOTHER_JACOBI, 2)
    it1, rel1, _ = S.pcg(A, b, lambda r: S.precondition(lin, r), 1e-8, bound)
    assert rel1 > 1e-8, (it1, rel1)


def test_options_strength_default_and_layout():
    assert amg.FullOptions.strength.offset == C.sizeof(amg.Options) and C.sizeof(amg.Options) % 8 == 0
    o = amg.FullOptions()
    amg.lib().amgb_options_default(C.byref(o))
    assert o.strength == 0.08 and o.lines == amg.LINES_X and o.transfer == amg.TRANSFER_LINEAR
    assert amg.SmoothedAggregation(4).strength == 0.08 and amg.SmoothedAggregation(4, 0.25).strength == 0.25
    with pytest.raises(NotImplementedError):
        amg.SmoothedAggregation(4).make_operators(100, 25, 0)
