"""Smoothed-aggregation coarsening (TRANSFER_SMOOTHED_AGGREGATION) on the device against its CPU oracle
(tests/oracle_sa.py): level operators and prolongators, per-level iterates of whole V-cycles, the
stand-alone transfers, iteration counts, PCG, the rejections, and PCG at 4097^2."""
import importlib

import numpy as np
import pytest
import scipy.sparse as sp

import oracle as O
import oracle_sa as S

amg = importlib.import_module("algebraic-multigrid_b200")
pytestmark = pytest.mark.gpu

CAP = 25  # n_levels is a cap: the hierarchy stops at <= 200 rows

SMOOTHERS = {
    "jacobi": (lambda: amg.DampedJacobi(2.0 / 3.0, 2), O.SMOOTHER_JACOBI, 2),
    "color_gs": (lambda: amg.MulticolorGaussSeidel(1), O.SMOOTHER_COLOR_GS, 1),
    "gs_auto": (lambda: amg.SparseGaussSeidel(mode=amg.GS_AUTO), O.SMOOTHER_GS, 1),
}

PROBLEMS = {
    "iso129": lambda: O.laplacian(129),
    "eps1e-3_129": lambda: O.laplacian(129, 1e-3),
    "eps1e3_65": lambda: O.laplacian(65, 1e3),
    "rect70x31": lambda: S.rectangular_poisson(70, 31),
    "perm65": lambda: S.permuted_laplacian(65, seed=3)[0],
    "lognormal65": lambda: S.lognormal_diffusion(65, seed=5),
}


def rhs(A):
    return np.random.default_rng(A.rows).standard_normal(A.rows)


def pair(Ao, smoother, b=None, every=10, n_iters=100, tol=1e-9, theta=0.08, **kw):
    make, kind, iters = SMOOTHERS[smoother]
    b = rhs(Ao) if b is None else b
    A = amg.CscMatrix(Ao.rows, Ao.cols, *Ao.arrays())
    interp = amg.SmoothedAggregation(CAP, theta)
    mg = amg.Multigrid(interp, make(), A, b, CAP, tol, every, n_iters, **kw)
    mo = S.Multigrid(Ao, b, CAP, tol, every, n_iters, kind, iters, 2.0 / 3.0, theta)
    return mg, mo, interp


def same_bytes(a, b):
    return np.asarray(a).tobytes() == np.asarray(b).tobytes()


def same_csc(M, Mo):
    c, r, v = Mo.arrays()
    return (np.array_equal(M.colptr, c) and np.array_equal(M.rowidx, r) and same_bytes(M.val, v))


@pytest.mark.parametrize("name", sorted(PROBLEMS))
def test_levels_operators_and_prolongators_match_oracle(name):
    mg, mo, interp = pair(PROBLEMS[name](), "jacobi")
    assert mg.transfer() == amg.TRANSFER_SMOOTHED_AGGREGATION
    assert mg.n_levels == mo.n_levels >= 2 and mg.get_n_dofs(mg.n_levels - 1) <= 200
    for l in range(mg.n_levels):
        assert mg.get_n_dofs(l) == mo.n_dofs(l)
        assert same_csc(mg.get_coefficient_matrix(l), mo.A(l)), ("A", l)
    for l in range(mg.n_levels - 1):
        assert same_csc(mg.get_transfer(l), mo.P(l)), ("P", l)
        assert same_csc(interp.get_P(l), mo.P(l)) and same_csc(interp.get_R(l), mo.R(l)), l


@pytest.mark.parametrize("name", sorted(PROBLEMS))
@pytest.mark.parametrize("smoother", ["jacobi", "color_gs", "gs_auto"])
def test_two_vcycles_bit_exact_per_level(name, smoother):
    mg, mo, _ = pair(PROBLEMS[name](), smoother)
    for _ in range(2):
        mg.vcycle()
        mo.vcycle()
        for l in range(mg.n_levels):
            assert same_bytes(mg.get_rhs(l), mo.f(l)), ("f", l)
            assert same_bytes(mg.get_soln(l), mo.u(l)), ("u", l)


@pytest.mark.parametrize("name", ["iso129", "perm65", "lognormal65"])
def test_fast_arithmetic_within_1e12(name):
    mg, mo, _ = pair(PROBLEMS[name](), "jacobi", arith=amg.ARITH_FAST)
    for _ in range(2):
        mg.vcycle()
        mo.vcycle()
    for l in range(mg.n_levels):
        u, uo = mg.get_soln(l), mo.u(l)
        assert np.linalg.norm(u - uo) <= 1e-12 * np.linalg.norm(uo), l


@pytest.mark.parametrize("name", ["iso129", "rect70x31", "perm65"])
def test_standalone_transfers_bit_exact(name):
    mg, mo, _ = pair(PROBLEMS[name](), "jacobi")
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
    assert mg.time_kernel(0, 2) > 0 and mg.time_kernel(0, 3) > 0


@pytest.mark.parametrize("m", [129, 257])
@pytest.mark.parametrize("smoother", ["jacobi", "gs_auto"])
def test_iteration_counts_equal_oracle(m, smoother):
    Ao, b = O.laplacian(m), O.rhs(m)
    tol = (1e-8 * np.linalg.norm(b)) ** 2  # rss criterion of solve()
    mg, mo, _ = pair(Ao, smoother, b, every=1, n_iters=200, tol=tol)
    mg.solve()
    mo.solve()
    assert mg.iters_done == mo.iters_done < 200


PCG = {
    "iso129": lambda: O.laplacian(129),
    "iso257": lambda: O.laplacian(257),
    "eps1e-3_257": lambda: O.laplacian(257, 1e-3),
    "rect300x120": lambda: S.rectangular_poisson(300, 120),
    "perm257": lambda: S.permuted_laplacian(257)[0],
    "lognormal129": lambda: S.lognormal_diffusion(129),
}


@pytest.mark.parametrize("name", sorted(PCG))
def test_pcg_within_one_iteration_of_oracle(name):
    Ao = PCG[name]()
    b = rhs(Ao)
    mg, mo, _ = pair(Ao, "jacobi", b, every=1, n_iters=100)
    mg.solve_pcg(1e-8, 100)
    mo.solve_pcg(b, 1e-8, 100)
    assert mg.last_error <= 1e-8 and mo.last_error <= 1e-8
    assert abs(mg.iters_done - mo.iters_done) <= 1, (mg.iters_done, mo.iters_done)


def test_rejections():
    A = amg.Grid.laplacian(64)
    b = amg.Grid.rhs(64)
    comm = amg.Comm(0, 1, lambda raw: raw)
    with pytest.raises(ValueError, match="sharded"):
        amg.Multigrid(amg.SmoothedAggregation(5), amg.DampedJacobi(), A, b, 5, comm=comm)
    with pytest.raises(ValueError, match="line Gauss-Seidel"):
        amg.Multigrid(amg.SmoothedAggregation(5), amg.LineGaussSeidel(), A, b, 5)
    with pytest.raises(ValueError, match="strength"):
        amg.Multigrid(amg.SmoothedAggregation(5, strength=-1.0), amg.DampedJacobi(), A, b, 5)
    D = sp.diags(np.arange(1.0, 301.0), format="csc")
    Dm = amg.CscMatrix(300, 300, D.indptr, D.indices, D.data)
    with pytest.raises(ValueError, match="level 0 does not reduce"):
        amg.Multigrid(amg.SmoothedAggregation(3), amg.DampedJacobi(), Dm, np.ones(300), 3)
    L = amg.Grid.laplacian(20).to_scipy().tolil()
    L[37, 37] = 0.0
    Z = sp.csc_matrix(L)
    Z.sort_indices()
    Zm = amg.CscMatrix(400, 400, Z.indptr, Z.indices, Z.data)
    with pytest.raises(ValueError, match="level 0 has a zero diagonal at row 37"):
        amg.Multigrid(amg.SmoothedAggregation(3), amg.DampedJacobi(), Zm, np.ones(400), 3)
    with pytest.raises(NotImplementedError):
        amg.SmoothedAggregation(3).make_operators(400, 100, 0)
    # fuse bits 1-7 do not apply: per-operator cycle
    mg = amg.Multigrid(amg.SmoothedAggregation(CAP), amg.DampedJacobi(2.0 / 3.0, 2), A, b, CAP)
    assert all(not mg.fused_legs(l) for l in range(mg.n_levels))
    assert mg.tail_first() == -1 and mg.mid_range()[0] == -1


def test_coarse_level_that_does_not_reduce_ends_the_hierarchy():
    """Poisson 129^2 with strength 0.15: level 5 (321 rows) has only weak couplings and is the coarsest."""
    Ao = O.laplacian(129)
    b = rhs(Ao)
    mg, mo, interp = pair(Ao, "jacobi", b, every=1, theta=0.15)
    assert mg.n_levels == mo.n_levels == 6 and mg.get_n_dofs(5) == mo.n_dofs(5) > 200
    for l in range(6):
        assert same_csc(mg.get_coefficient_matrix(l), mo.A(l)), l
    assert same_csc(interp.get_P(4), mo.P(4))
    for _ in range(2):
        mg.vcycle()
        mo.vcycle()
    for l in range(6):
        assert same_bytes(mg.get_soln(l), mo.u(l)), l
    mg.set_soln(0, np.zeros(Ao.rows))
    mg.solve_pcg(1e-8, 100)
    assert mg.last_error <= 1e-8


def big_problem(kind, m):
    if kind == "perm":
        L = O.laplacian(m).to_scipy()
        perm = np.random.default_rng(0).permutation(m * m)
        M = sp.csc_matrix(L[perm][:, perm])
        M.sort_indices()
        return M
    A = amg.Grid.laplacian(m, 1e-3 if kind == "aniso" else 1.0)
    return A.to_scipy()


@pytest.mark.parametrize("kind", ["iso", "aniso", "perm"])
def test_4097_pcg_reaches_1e8(kind):
    m = 4097
    M = big_problem(kind, m)
    b = np.random.default_rng(11).standard_normal(m * m)
    A = amg.CscMatrix(m * m, m * m, M.indptr, M.indices, M.data)
    # the Galerkin levels turn dense above 200 rows here: the first one that does not reduce is the coarsest
    mg = amg.Multigrid(amg.SmoothedAggregation(CAP), amg.DampedJacobi(2.0 / 3.0, 2), A, b, CAP, 1e-9, 1, 100,
                       arith=amg.ARITH_FAST)
    mg.solve_pcg(1e-8, 100)
    u = mg.get_soln(0)
    rel = np.linalg.norm(b - M @ u) / np.linalg.norm(b)
    assert mg.last_error <= 1e-8 and rel <= 1.01e-8, (mg.iters_done, rel)
