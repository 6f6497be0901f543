"""Smoothed aggregation without a GPU on the matrix families of tests/sa_matrices.py (9-point, 3-D 7- and
27-point, P1 finite elements, arrowhead, convection-diffusion, negated Laplacian, Dirichlet rows, signed
zeros): amgb_sa_aggregate and the host setup of host_setup.cpp against the numpy oracle, byte for byte;
the level sizes of the Dirichlet and strength-0 hierarchies; the 27-point rejection at the default
strength; and that the families reach the global-memory tables of the device product."""
import importlib

import numpy as np
import pytest
import scipy.sparse as sp

import oracle as O
import oracle_sa as S
import sa_matrices as G
from test_sa_host import as_amg, host_levels, same_bytes

amg = importlib.import_module("algebraic-multigrid_b200")

# the small size of every family, and the size the GPU tests compare with the oracle
SIZES = {"nine": (65, 129), "p7": (13, 21), "q1_27": (11, 17), "p1fe": (3000, 20000), "arrow": (33, 65),
         "conv": (65, 129), "neg": (65, 129), "dir": (33, 65), "dirsym": (33, 65), "zeros": (65, 129)}
CASES = [(name, n) for name in sorted(SIZES) for n in SIZES[name]]


def family(name, n):
    gen, theta, _ = G.FAMILIES[name]
    return gen(n), theta


def assert_host_matches_oracle(A, theta):
    As, Ps, _, _ = S.build(A, 25, theta)
    hA, hP = host_levels(A, 25, theta)
    assert len(hA) == len(As) >= 2 and len(hP) == len(Ps)
    for kind, host, oracle in (("A", hA, As), ("P", hP, Ps)):
        for l, M in enumerate(oracle):
            c, r, v = M.arrays()
            assert np.array_equal(host[l][0], c) and np.array_equal(host[l][1], r), (kind, l)
            assert same_bytes(host[l][2], v), (kind, l)
    return As, Ps


@pytest.mark.parametrize("name,n", CASES)
def test_aggregate_matches_oracle(name, n):
    A, theta = family(name, n)
    agg, k = amg.sa_aggregate(as_amg(A), theta)
    agg_o, k_o, _ = S.aggregate(A, theta)
    assert k == k_o and 0 < k < A.rows
    np.testing.assert_array_equal(agg, agg_o)


@pytest.mark.parametrize("name,n", CASES)
def test_host_setup_bit_identical_to_oracle(name, n):
    A, theta = family(name, n)
    assert_host_matches_oracle(A, theta)


def test_generators_are_sorted_seeded_and_keep_signed_zeros():
    for name, (gen, _, symmetric) in sorted(G.FAMILIES.items()):
        A = gen(SIZES[name][0])
        c, r, v = A.arrays()
        assert all((np.diff(r[c[j]:c[j + 1]]) > 0).all() for j in range(A.cols)), name
        M = A.to_scipy()
        if symmetric:  # in value
            assert abs(M - M.T).max() == 0.0, name
        else:
            assert abs(M - M.T).max() > 0.0, name
    a, b = G.p1_fe(3000, seed=4), G.p1_fe(3000, seed=4)
    assert all(same_bytes(x, y) for x, y in zip(a.arrays(), b.arrays()))
    v = G.signed_zeros(65).arrays()[2]
    assert (v == 0).sum() > 1000 and np.signbit(v[v == 0]).sum() > 500 and (~np.signbit(v[v == 0])).sum() > 500
    # symmetric in value, not in bits: the transpose swaps some +0 and -0
    Z = G.signed_zeros(65)
    assert not same_bytes(Z.arrays()[2], Z.transpose().arrays()[2])


def test_q1_27_needs_a_strength_below_the_default():
    A = G.q1_27(17)
    with pytest.raises(ValueError, match="level 0 does not reduce") as host:
        host_levels(A, 25, 0.08)
    with pytest.raises(ValueError, match="level 0 does not reduce") as oracle:
        S.build(A, 25, 0.08)
    assert str(host.value) == str(oracle.value) + " (4913 rows, 4913 aggregates)"
    assert [M.rows for M in S.build(A, 25, 0.04)[0]] == [4913, 360, 160]


@pytest.mark.parametrize("sym,sizes", [(True, [4225, 943, 362, 283, 266]), (False, [4225, 811, 123])])
def test_dirichlet_level_sizes(sym, sizes):
    """Boundary rows set to identity rows are isolated: with symmetric elimination they stay singletons on
    every level, until a level that does not reduce (266 rows, above the 200-row target) is the coarsest."""
    A = G.dirichlet(65, sym)
    As, _ = assert_host_matches_oracle(A, 0.08)
    assert [M.rows for M in As] == sizes
    agg, k = amg.sa_aggregate(as_amg(As[-1]))
    assert (k == As[-1].rows) == sym


@pytest.mark.parametrize("name,make,sizes", [
    ("laplacian65", lambda: O.laplacian(65), [4225, 726, 88]),
    ("nine65", lambda: G.nine_point(65), [4225, 484, 64]),
])
def test_strength_zero(name, make, sizes):
    """theta = 0: every non-zero off-diagonal entry is strong."""
    As, _ = assert_host_matches_oracle(make(), 0.0)
    assert [M.rows for M in As] == sizes


def test_the_oracle_sized_families_reach_the_global_tables():
    """Columns of A P and R (A P) whose product bound exceeds 512 go to the global-memory tables of the
    device product; per level, (A P, R (A P))."""
    expect = {
        ("p7", 21): [(0, 0), (779, 1029), (111, 0)],
        ("q1_27", 17): [(358, 0), (0, 0)],
        ("p1fe", 20000): [(0, 1), (423, 0), (0, 0)],
        ("arrow", 65): [(727, 727), (106, 0)],
        ("zeros", 129): [(0, 0), (0, 1813), (240, 0), (0, 0)],
    }
    for (name, n), counts in expect.items():
        A, theta = family(name, n)
        As, Ps, _, _ = S.build(A, 25, theta)
        assert G.global_table_columns(As, Ps) == counts, name


def test_product_bounds_match_a_direct_count():
    rng = np.random.default_rng(0)
    L = sp.random(50, 40, density=0.2, format="csc", random_state=rng)
    R = sp.random(40, 30, density=0.1, format="lil", random_state=rng)
    R[:, 3] = 0.0
    R = sp.csc_matrix(R)
    Lc = np.diff(L.indptr)
    direct = [min(50, int(sum(Lc[k] for k in R.indices[R.indptr[j]:R.indptr[j + 1]]))) for j in range(30)]
    assert G.product_bounds(L, R).tolist() == direct and direct[3] == 0

