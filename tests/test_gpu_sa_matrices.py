"""Smoothed aggregation on the device for the matrix families of tests/sa_matrices.py: 9-point, 3-D 7- and
27-point, P1 finite elements on a Delaunay mesh, an arrowhead with a dense row and column, upwind
convection-diffusion, the negated Laplacian, Dirichlet rows (symmetric and unsymmetric elimination) and
explicit signed zeros.  These reach what the five-point families do not: products whose columns take the
global-memory hash tables, SELL rows hundreds of entries long in the level operators and in R, the
unsymmetric rows mirror of the device-resident Jacobi path, isolated rows and mixed-sign diagonals.

At sizes the numpy oracle (tests/oracle_sa.py) handles, the device-built levels and P, two V-cycles per
level, the stand-alone transfers, solve() and PCG are checked against it; at larger sizes the device setup
is checked against the host setup (AMGB_HOST_SETUP=1).  amgb_csc_multiply is checked at the edges of its
hash tables against host_setup.cpp's product and against an exact order-free reference."""
import functools
import importlib

import numpy as np
import pytest
import scipy.sparse as sp

import oracle as O
import oracle_sa as S
import sa_matrices as G
from test_gpu_sa_device_setup import host_multiply, same_csc

amg = importlib.import_module("algebraic-multigrid_b200")
pytestmark = pytest.mark.gpu

CAP = 25

SMOOTHERS = {
    "jacobi": (lambda: amg.DampedJacobi(2.0 / 3.0, 2), O.SMOOTHER_JACOBI, 2),
    "color_gs": (lambda: amg.MulticolorGaussSeidel(1), O.SMOOTHER_COLOR_GS, 1),
    "gs_auto": (lambda: amg.SparseGaussSeidel(mode=amg.GS_AUTO), O.SMOOTHER_GS, 1),
}

# the size of every family that the oracle checks (tests/test_sa_matrices_host.py pins which of them reach
# the global-memory tables)
ORACLE_SIZE = {"nine": 129, "p7": 21, "q1_27": 17, "p1fe": 20000, "arrow": 65, "conv": 129, "neg": 129,
               "dir": 65, "dirsym": 65, "zeros": 129}
NAMES = sorted(ORACLE_SIZE)
SYMMETRIC = [name for name in NAMES if G.FAMILIES[name][2]]


@functools.lru_cache(maxsize=None)
def problem(name, n=None):
    gen, theta, _ = G.FAMILIES[name]
    return gen(ORACLE_SIZE[name] if n is None else n), theta


def rhs(rows):
    return np.random.default_rng(rows).standard_normal(rows)


def as_amg(Ao):
    return amg.CscMatrix(Ao.rows, Ao.cols, *Ao.arrays())


def pair(name, smoother, b=None, every=10, n_iters=100, tol=1e-9, **kw):
    Ao, theta = problem(name)
    make, kind, iters = SMOOTHERS[smoother]
    b = rhs(Ao.rows) if b is None else b
    interp = amg.SmoothedAggregation(CAP, theta)
    mg = amg.Multigrid(interp, make(), as_amg(Ao), b, CAP, tol, every, n_iters, **kw)
    mo = S.Multigrid(Ao, b, CAP, tol, every, n_iters, kind, iters, 2.0 / 3.0, theta)
    return mg, mo, interp


def same_bytes(a, b):
    return np.asarray(a).tobytes() == np.asarray(b).tobytes()


def same_as_oracle(M, Mo):
    c, r, v = Mo.arrays()
    return M.rows == Mo.rows and M.cols == Mo.cols and same_bytes(M.colptr, c) and same_bytes(M.rowidx, r) \
        and same_bytes(M.val, v)


def build(A, smoother, theta, monkeypatch, host):
    if host:
        monkeypatch.setenv("AMGB_HOST_SETUP", "1")
    else:
        monkeypatch.delenv("AMGB_HOST_SETUP", raising=False)
    try:
        return amg.Multigrid(amg.SmoothedAggregation(CAP, theta), SMOOTHERS[smoother][0](), A, rhs(A.rows), CAP,
                             1e-9, 10, 100)
    finally:
        monkeypatch.delenv("AMGB_HOST_SETUP", raising=False)


def assert_device_matches_host(A, theta, smoother, monkeypatch, cycles=2):
    dev = build(A, smoother, theta, monkeypatch, host=False)
    ref = build(A, smoother, theta, monkeypatch, host=True)
    assert dev.device_setup and not ref.device_setup
    L = dev.n_levels
    assert L == ref.n_levels >= 2
    for l in range(L):
        assert dev.get_n_dofs(l) == ref.get_n_dofs(l), l
        assert dev.format(l) == ref.format(l), l
        assert dev.nnz(l) == ref.nnz(l) and dev.nnz_device(l) == ref.nnz_device(l), l
        assert same_csc(dev.get_coefficient_matrix(l), ref.get_coefficient_matrix(l)), ("A", l)
    for l in range(L - 1):
        assert same_csc(dev.get_transfer(l), ref.get_transfer(l)), ("P", l)
    assert dev.vcycle_bytes() == ref.vcycle_bytes()
    for _ in range(cycles):
        dev.vcycle()
        ref.vcycle()
        for l in range(L):
            assert same_bytes(dev.get_rhs(l), ref.get_rhs(l)), ("f", l)
            assert same_bytes(dev.get_soln(l), ref.get_soln(l)), ("u", l)


# ---- against the oracle ----
@pytest.mark.parametrize("name", NAMES)
def test_levels_and_prolongators_match_oracle(name):
    mg, mo, interp = pair(name, "jacobi")
    assert mg.device_setup
    assert mg.n_levels == mo.n_levels >= 2
    for l in range(mg.n_levels):
        assert mg.get_n_dofs(l) == mo.n_dofs(l), l
        assert same_as_oracle(mg.get_coefficient_matrix(l), mo.A(l)), ("A", l)
    for l in range(mg.n_levels - 1):
        assert same_as_oracle(mg.get_transfer(l), mo.P(l)), ("P", l)
        assert same_as_oracle(interp.get_P(l), mo.P(l)) and same_as_oracle(interp.get_R(l), mo.R(l)), l


@pytest.mark.parametrize("name", NAMES)
@pytest.mark.parametrize("smoother", ["jacobi", "gs_auto"])
def test_formats_and_entry_counts_match_host_setup(name, smoother, monkeypatch):
    Ao, theta = problem(name)
    dev = build(as_amg(Ao), smoother, theta, monkeypatch, host=False)
    ref = build(as_amg(Ao), smoother, theta, monkeypatch, host=True)
    assert dev.device_setup and not ref.device_setup and dev.n_levels == ref.n_levels
    for l in range(dev.n_levels):
        assert dev.format(l) == ref.format(l), l
        assert dev.nnz(l) == ref.nnz(l) and dev.nnz_device(l) == ref.nnz_device(l), l
    assert dev.vcycle_bytes() == ref.vcycle_bytes()


def line_scan_levels(mg):
    """Levels whose GS_AUTO sweep runs the line-scan kernel: banded operators that are not 2-D grid
    operators (the 3-D stencils).  It re-associates the distance-1 chain (<= 1e-14 relative per sweep,
    include/amgb.h), so it is not the reference's arithmetic bit for bit."""
    return [l for l in range(mg.n_levels) if mg.gs_kernel(l) == amg.GS_KERNEL_LINESCAN]


@pytest.mark.parametrize("name", NAMES)
@pytest.mark.parametrize("smoother", sorted(SMOOTHERS))
def test_two_vcycles_bit_exact_per_level(name, smoother):
    mg, mo, _ = pair(name, smoother)
    scan = line_scan_levels(mg) if smoother == "gs_auto" else []
    if (name, smoother) == ("p7", "gs_auto"):
        assert scan  # the 7-point level 0
    for _ in range(2):
        mg.vcycle()
        mo.vcycle()
        for l in range(mg.n_levels):
            if scan:
                for v, vo in ((mg.get_rhs(l), mo.f(l)), (mg.get_soln(l), mo.u(l))):
                    assert np.linalg.norm(v - vo) <= 1e-12 * np.linalg.norm(vo), l
                continue
            assert same_bytes(mg.get_rhs(l), mo.f(l)), ("f", l)
            assert same_bytes(mg.get_soln(l), mo.u(l)), ("u", l)


# P1 FE on random points is ill-conditioned (PCG takes 79 iterations): the FMA roundings of fast arithmetic
# grow to 3.5e-12 relative on its level 1 within two cycles
FAST_TOL = {"p1fe": 1e-11}


@pytest.mark.parametrize("name", NAMES)
def test_fast_arithmetic_within_1e12(name):
    mg, mo, _ = pair(name, "jacobi", arith=amg.ARITH_FAST)
    for _ in range(2):
        mg.vcycle()
        mo.vcycle()
    for l in range(mg.n_levels):
        u, uo = mg.get_soln(l), mo.u(l)
        assert np.linalg.norm(u - uo) <= FAST_TOL.get(name, 1e-12) * np.linalg.norm(uo), l


@pytest.mark.parametrize("name", NAMES)
def test_standalone_transfers_bit_exact(name):
    mg, mo, _ = pair(name, "jacobi")
    rng = np.random.default_rng(7)
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


# solve() to 1e-8 relative: the cycles it takes on the oracle (None: still above after 200 cycles).  The
# unsymmetric families diverge: convection-diffusion grows without bound, and with Gauss-Seidel the
# unsymmetric Dirichlet problem overflows to a NaN rss at cycle 123, which ends solve() (NaN > tol is false)
SOLVE_ITERS = {
    ("nine", "jacobi"): 25, ("nine", "gs_auto"): 18,
    ("p7", "jacobi"): 16, ("p7", "gs_auto"): 10,
    ("q1_27", "jacobi"): 13, ("q1_27", "gs_auto"): 8,
    ("p1fe", "jacobi"): None, ("p1fe", "gs_auto"): None,
    ("arrow", "jacobi"): 21, ("arrow", "gs_auto"): 13,
    ("conv", "jacobi"): None, ("conv", "gs_auto"): None,
    ("neg", "jacobi"): 28, ("neg", "gs_auto"): 18,
    ("dir", "jacobi"): 73, ("dir", "gs_auto"): 123,
    ("dirsym", "jacobi"): 21, ("dirsym", "gs_auto"): 14,
    ("zeros", "jacobi"): 11, ("zeros", "gs_auto"): 6,
}


@pytest.mark.parametrize("name", NAMES)
@pytest.mark.parametrize("smoother", ["jacobi", "gs_auto"])
def test_solve_iteration_counts_equal_oracle(name, smoother):
    b = rhs(problem(name)[0].rows)
    tol = (1e-8 * np.linalg.norm(b)) ** 2  # rss criterion of solve()
    mg, mo, _ = pair(name, smoother, b, every=1, n_iters=200, tol=tol)
    mg.solve()
    mo.solve()
    assert mg.iters_done == mo.iters_done == (SOLVE_ITERS[name, smoother] or 200)
    if (name, smoother) == ("dir", "gs_auto"):
        assert np.isnan(mg.last_error) and np.isnan(mo.last_error)
        return
    # bit-exact iterates; the rss reductions differ in order (and the line-scan sweeps of p7 re-associate)
    tol = 1e-6 if line_scan_levels(mg) else 1e-12
    assert abs(mg.last_error - mo.last_error) <= tol * abs(mo.last_error), (mg.last_error, mo.last_error)


@pytest.mark.parametrize("name", SYMMETRIC)
def test_pcg_reaches_1e8(name):
    Ao, _ = problem(name)
    b = rhs(Ao.rows)
    mg, mo, _ = pair(name, "jacobi", b, every=1, n_iters=100)
    mg.solve_pcg(1e-8, 100)
    mo.solve_pcg(b, 1e-8, 100)
    assert mg.last_error <= 1e-8 and mo.last_error <= 1e-8
    assert abs(mg.iters_done - mo.iters_done) <= 1, (mg.iters_done, mo.iters_done)
    rel = np.linalg.norm(b - Ao.to_scipy() @ mg.get_soln(0)) / np.linalg.norm(b)
    assert rel <= 1.05e-8, (mg.iters_done, rel)


# ---- device setup against host setup, at sizes the oracle is too slow for ----
# (the arrowhead's products are dense: test_arrowhead_513_product_exceeds_int32_indexing)
LARGE = {"p7_65": ("p7", 65), "q1_27_41": ("q1_27", 41), "p1fe_300k": ("p1fe", 300_000), "conv1025": ("conv", 1025)}


@pytest.mark.parametrize("case", sorted(LARGE))
def test_large_levels_and_vcycles_match_host_setup(case, monkeypatch):
    Ao, theta = problem(*LARGE[case])
    assert_device_matches_host(as_amg(Ao), theta, "jacobi", monkeypatch)


def test_arrowhead_513_product_exceeds_int32_indexing(monkeypatch):
    """The dense row of the arrowhead makes row 0 of P dense, so A P is dense: 263,169 rows times some 45,000
    aggregates at 513^2, beyond int32 indexing.  The device setup reports the host's overflow error."""
    Ao, theta = problem("arrow", 513)
    with pytest.raises(amg.AmgbError, match="multiply: result exceeds int32 indexing"):
        build(as_amg(Ao), "jacobi", theta, monkeypatch, host=False)


# ---- amgb_csc_multiply at the edges of its hash tables ----
def small_ints(rng, size, zeros=True):
    """|v| <= 8, so every product and sum below is exact; zeros=True stores some +0 and -0."""
    v = rng.integers(-8, 9, size=size).astype(np.float64)
    if zeros:
        v[rng.random(size) < 0.05] = -0.0
    else:
        v[v == 0] = 1.0
    return v


def csc(rows, cols, colptr, rowidx, val):
    return amg.CscMatrix(rows, cols, np.asarray(colptr), np.asarray(rowidx), np.asarray(val))


def from_columns(rows, columns, rng, zeros=True):
    """CSC with the given row lists per column (sorted here) and small-integer values."""
    colptr = np.concatenate([[0], np.cumsum([len(c) for c in columns])]).astype(np.int64)
    rowidx = np.concatenate([np.sort(np.asarray(c, np.int64)) for c in columns]) if colptr[-1] else np.zeros(0, np.int64)
    return csc(rows, len(columns), colptr, rowidx, small_ints(rng, int(colptr[-1]), zeros))


def assert_exact_product(A, B):
    """C = csc_multiply(A, B) equals the host product byte for byte, and an order-free reference: its pattern
    is the product of the 0/1 structures, its values equal scipy's A @ B wherever scipy keeps an entry (all
    sums are exact) and are exactly zero elsewhere (scipy drops computed zeros; the library keeps them)."""
    C = amg.csc_multiply(A, B)
    assert same_csc(C, host_multiply(A, B))
    assert C.rows == A.rows and C.cols == B.cols
    Cs = C.to_scipy()
    pattern = sp.csc_matrix(G.structure(A.to_scipy()) @ G.structure(B.to_scipy()))
    pattern.sort_indices()
    assert np.array_equal(C.colptr, pattern.indptr) and np.array_equal(C.rowidx, pattern.indices)
    ref = sp.csc_matrix(A.to_scipy() @ B.to_scipy())
    assert ref.nnz <= C.nnz
    assert (Cs - ref).count_nonzero() == 0  # exact sums: equal on scipy's pattern, zeros elsewhere
    return C


def test_csc_multiply_bound_512_and_513():
    """Column bounds of exactly 512 (shared table: 1024 slots) and 513 (global table), with L columns
    longer than 32 so the lanes loop within a step; and bounds clipped by L.rows on either side."""
    rng = np.random.default_rng(0)
    m = 2000
    lens = [512, 1, 40, 33, 300, 212, 7]
    A = from_columns(m, [rng.choice(m, size=n, replace=False) for n in lens], rng)
    # bounds 512, 513, 585, 8, 0 (empty), 1104, 512 (300 + 212), 40
    B = from_columns(len(lens), [[0], [0, 1], [2, 3, 4, 5], [1, 6], [], [0, 2, 3, 4, 5, 6], [4, 5], [2]], rng)
    bounds = G.product_bounds(A.to_scipy(), B.to_scipy())
    assert 512 in bounds and 513 in bounds and (bounds > 513).any() and 0 in bounds
    assert_exact_product(A, B)
    # the same columns over 600 rows (bound 513.. clipped to 600: global) and 300 rows (clipped to 300: shared)
    for rows in (600, 300):
        A2 = from_columns(rows, [rng.choice(rows, size=min(n, rows), replace=False) for n in lens], rng)
        bounds = G.product_bounds(A2.to_scipy(), B.to_scipy())
        assert bounds.max() == rows
        assert_exact_product(A2, B)


@pytest.mark.parametrize("m,k,n", [(0, 3, 2), (3, 0, 2), (3, 2, 0), (0, 0, 0), (1, 1, 1), (1, 5, 1), (5, 1, 5),
                                   (1, 700, 3), (700, 1, 3)])
def test_csc_multiply_degenerate_shapes(m, k, n):
    rng = np.random.default_rng(m * 10000 + k * 100 + n)
    A = from_columns(m, [rng.choice(m, size=rng.integers(0, m + 1), replace=False) if m else [] for _ in range(k)], rng)
    B = from_columns(k, [rng.choice(k, size=rng.integers(0, k + 1), replace=False) if k else [] for _ in range(n)], rng)
    assert_exact_product(A, B)


def test_csc_multiply_more_wide_columns_than_global_warps():
    """200 columns with bounds from 1,500 to 300,000 over a 300,000-row L: the 1 GiB budget of per-warp
    global tables of 2^20 slots (12 MiB) allows 85 warps, rounded up to 88, so warps loop over the listed
    columns and reuse their tables for columns of smaller and of larger capacity.  L's columns share a pool
    of 3,000 rows, so the product columns stay small while their bounds are large."""
    rng = np.random.default_rng(5)
    m, K = 300_000, 200
    pool = rng.choice(m, size=3000, replace=False)
    A = from_columns(m, [rng.choice(pool, size=1500, replace=False) for _ in range(K)], rng, zeros=False)
    counts = np.concatenate([[K], rng.integers(1, K + 1, size=K - 1)])  # one column reaches 300,000
    cols = [rng.choice(K, size=c, replace=False) for c in counts]
    cols += [[], [3], rng.choice(K, size=2, replace=False)]  # empty, and two columns of bound <= 3,000
    B = from_columns(K, cols, rng, zeros=False)
    bounds = G.product_bounds(A.to_scipy(), B.to_scipy())
    assert bounds.max() == m and (bounds > 512).sum() >= 200
    assert_exact_product(A, B)
