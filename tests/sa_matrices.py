"""Matrix families for smoothed aggregation beyond the 2-D five-point stencil.  TEST INFRASTRUCTURE ONLY.

Every generator takes a size, uses numpy / scipy only and returns an oracle Csc (tests/oracle_sa.py) with
ascending row indices; random ones take a seed.  Whatever entries the scipy assembly stores are kept
(no eliminate_zeros), so explicit zeros pass through unchanged.

  nine_point(m)           9-point Q1 stiffness on an m x m grid: kron(K, M) + kron(M, K)
  poisson7(k)             3-D 7-point Laplacian on a k^3 grid
  q1_27(k)                3-D 27-point Q1 stiffness: kron(K, M, M) + kron(M, K, M) + kron(M, M, K); its edge
                          and corner couplings are weak at the default strength 0.08, so it wants about 0.04
  p1_fe(n, seed)          P1 finite elements on a Delaunay mesh of n seeded random points, plus 1e-3 I
  arrowhead(m)            Grid::laplacian(m) plus a dense first row and column
  convection(m, pe)       upwind convection-diffusion, unsymmetric
  negated_laplacian(m)    -Grid::laplacian(m): a positive diagonal where Grid::laplacian's is negative
  dirichlet(m, sym)       Grid::laplacian(m) with the boundary rows set to identity rows; sym also clears
                          the boundary columns (symmetric elimination), else A is unsymmetric
  signed_zeros(m, seed)   nine_point(m) with a seeded share of its off-diagonal pairs stored as explicit
                          +0.0 / -0.0 (signs drawn per entry: symmetric in value, not in bits)

K and M are the 1-D stiffness tridiag(-1, 2, -1) and mass tridiag(1, 4, 1) / 6.
"""
import numpy as np
import scipy.sparse as sp
import scipy.spatial as spt

import oracle as O
import oracle_sa as S


def _lap1(k):
    return sp.diags([-1.0, 2.0, -1.0], [-1, 0, 1], shape=(k, k))


def _mass1(k):
    return sp.diags([1.0, 4.0, 1.0], [-1, 0, 1], shape=(k, k)) / 6.0


def nine_point(m):
    K, M = _lap1(m), _mass1(m)
    return S._csc(sp.kron(K, M) + sp.kron(M, K))


def poisson7(k):
    I, L = sp.identity(k), _lap1(k)
    return S._csc(sp.kron(sp.kron(L, I), I) + sp.kron(sp.kron(I, L), I) + sp.kron(sp.kron(I, I), L))


def q1_27(k):
    K, M = _lap1(k), _mass1(k)
    return S._csc(sp.kron(sp.kron(K, M), M) + sp.kron(sp.kron(M, K), M) + sp.kron(sp.kron(M, M), K))


def p1_fe(n, seed=0):
    rng = np.random.default_rng(seed)
    X = rng.random((n, 2))
    T = spt.Delaunay(X).simplices
    P = X[T]  # (triangles, 3 vertices, 2)
    B = np.stack([P[:, 1] - P[:, 0], P[:, 2] - P[:, 0]], axis=2)  # columns: edge vectors
    area = np.abs(np.linalg.det(B)) / 2.0
    G = np.linalg.inv(B).transpose(0, 2, 1) @ np.array([[-1.0, 1.0, 0.0], [-1.0, 0.0, 1.0]])
    K = area[:, None, None] * (G.transpose(0, 2, 1) @ G)  # element stiffness, 3 x 3
    rows = np.repeat(T, 3, axis=1).ravel()
    cols = np.tile(T, (1, 3)).ravel()
    M = sp.csc_matrix((K.ravel(), (rows, cols)), shape=(n, n))
    return S._csc(M + 1e-3 * sp.identity(n))


def arrowhead(m):
    n = m * m
    L = O.laplacian(m).to_scipy().tocoo()
    keep = (L.row > 0) & (L.col > 0)
    edge = np.arange(1, n)
    rows = np.concatenate([L.row[keep], np.zeros(n - 1, np.int64), edge, [0]])
    cols = np.concatenate([L.col[keep], edge, np.zeros(n - 1, np.int64), [0]])
    vals = np.concatenate([L.data[keep], np.full(2 * (n - 1), -1e-2), [4.0 + 1e-2 * n]])
    return S._csc(sp.csc_matrix((vals, (rows, cols)), shape=(n, n)))


def convection(m, pe=10.0):
    I, D = sp.identity(m), _lap1(m)
    C = sp.diags([-1.0, 1.0], [-1, 0], shape=(m, m)) * (pe / m)
    return S._csc(sp.kron(D + C, I) + sp.kron(I, D))


def negated_laplacian(m):
    return S._csc(-O.laplacian(m).to_scipy())


def boundary_rows(m):
    i = np.arange(m * m)
    return i[(i % m == 0) | (i % m == m - 1) | (i // m == 0) | (i // m == m - 1)]


def dirichlet(m, sym):
    L = O.laplacian(m).to_scipy().tocoo()
    b = boundary_rows(m)
    on = np.zeros(m * m, bool)
    on[b] = True
    keep = ~on[L.row] & ~(sym & on[L.col])
    rows, cols = np.concatenate([L.row[keep], b]), np.concatenate([L.col[keep], b])
    vals = np.concatenate([L.data[keep], np.ones(b.size)])
    return S._csc(sp.csc_matrix((vals, (rows, cols)), shape=(m * m, m * m)))


def signed_zeros(m, seed=0, share=0.3):
    M = sp.csc_matrix(nine_point(m).to_scipy())
    M.sort_indices()
    rng = np.random.default_rng(seed)
    col = np.repeat(np.arange(M.shape[1]), np.diff(M.indptr))
    row = M.indices
    upper = np.flatnonzero(row < col)
    pick = upper[rng.random(upper.size) < share]
    # the mirrored entry (col, row) of each picked (row, col)
    mirror = M.indptr[row[pick]] + np.array([np.searchsorted(M.indices[M.indptr[r]:M.indptr[r + 1]], c)
                                             for r, c in zip(row[pick], col[pick])], np.int64)
    both = np.concatenate([pick, mirror])
    M.data[both] = np.where(rng.random(both.size) < 0.5, 0.0, -0.0)
    return O.Csc.from_arrays(M.shape[0], M.shape[1], M.indptr, M.indices, M.data)


# name -> (generator of one size argument, strength, symmetric in value)
FAMILIES = {
    "nine": (nine_point, 0.08, True),
    "p7": (poisson7, 0.08, True),
    "q1_27": (q1_27, 0.04, True),
    "p1fe": (p1_fe, 0.08, True),
    "arrow": (arrowhead, 0.08, True),
    "conv": (convection, 0.08, False),
    "neg": (negated_laplacian, 0.08, True),
    "dir": (lambda m: dirichlet(m, False), 0.08, False),
    "dirsym": (lambda m: dirichlet(m, True), 0.08, True),
    "zeros": (signed_zeros, 0.08, True),
}


def product_bounds(L, R):
    """k_spgemm_bound of L R on the CPU: per column j of R, min(L.rows, sum over R(:, j) of |L(:, k)|)."""
    cs = np.concatenate([[0], np.cumsum(np.diff(L.indptr).astype(np.int64)[R.indices])])
    return np.minimum(cs[R.indptr[1:]] - cs[R.indptr[:-1]], L.shape[0])


def structure(M):
    """The 0/1 structure of a CSC (explicit zeros count as entries)."""
    M = sp.csc_matrix(M, copy=True)
    M.data = np.ones_like(M.data)
    return M


def global_table_columns(As, Ps, small_bound=512):
    """Per level l: (columns of A_l P_l, columns of R_l (A_l P_l)) whose bound exceeds the shared table's
    small_bound, i.e. that the device setup's product sends to the global-memory tables."""
    out = []
    for A, P in zip(As, Ps):
        Al, Pl = structure(A.to_scipy()), structure(P.to_scipy())
        Rl = sp.csc_matrix(Pl.T)
        AP = sp.csc_matrix(Al @ Pl)  # positive entries only: scipy drops none
        out.append((int((product_bounds(Al, Pl) > small_bound).sum()), int((product_bounds(Rl, AP) > small_bound).sum())))
    return out
