"""CPU oracle of smoothed-aggregation coarsening (TRANSFER_SMOOTHED_AGGREGATION).  TEST INFRASTRUCTURE ONLY.

The transfer has no reference counterpart: this definition is the specification, mirrored in
include/amgb.h.  The hierarchy is composed from the CPU oracle's own operations (oracle/amg_oracle.c:
the transpose, Eigen's conservative product order, the residual, spmv, the three smoothers and the
banded LDL^T) exactly like tests/oracle_bilinear2d.py composes its own; only P differs.

"Row i" is CSC column i; sums start from +0 and run over ascending index.
  1. strength: j != i is a strong neighbour of i when |a_ij| > theta * sqrt(|a_ii| * |a_jj|) (product,
     then sqrt, then multiply); explicit zeros are never strong; a zero diagonal is an error.
  2. aggregation, ids in creation order:
     pass 1, i ascending: i and all its strong neighbours unaggregated -> they form a new aggregate
             (a node without strong neighbours becomes a singleton);
     pass 2, each remaining i ascending: joins the pass-1 aggregate of its first strong neighbour
             (ascending column) that pass 1 aggregated;
     pass 3, each still remaining i ascending: a new aggregate with its still unaggregated strong
             neighbours.
  3. tentative T(i, agg(i)) = 1.
  4. rho = max_i (sum_j |a_ij|) / |a_ii| over the stored entries, w = (4.0 / 3.0) / rho, c_i = w / a_ii;
     s_iJ = sum of a_ik over the stored k of row i with agg(k) = J;
     P(i, J) = T(i, J) - c_i * s_iJ (separate multiply and subtract) for every J row i touches,
     ascending; computed zeros are kept.
  5. R = P^T, A_H = galerkin(R, A, P).
  6. coarsen while l + 1 < n_levels and n_l > 200; a level l >= 1 whose aggregation does not reduce it is
     the coarsest level; when level 0 does not reduce, an error.
"""
import numpy as np

import oracle as O

MAX_COARSE = 200


def _rows(A):
    """(colptr, rowidx, val) of an oracle Csc or an amg CscMatrix."""
    if isinstance(A, O.Csc):
        return A.arrays()
    return np.asarray(A.colptr), np.asarray(A.rowidx), np.asarray(A.val)


def diagonal(colptr, rowidx, val, level=0):
    n = colptr.shape[0] - 1
    col = np.repeat(np.arange(n), np.diff(colptr))
    d = np.zeros(n)
    on = rowidx == col
    d[col[on]] = val[on]
    bad = np.flatnonzero(d == 0.0)
    if bad.size:
        raise ValueError("smoothed aggregation: level %d has a zero diagonal at row %d" % (level, bad[0]))
    return d


def strong(colptr, rowidx, val, theta, level=0):
    """Boolean mask over the stored entries: entry p (row i = its column, j = rowidx[p]) is strong."""
    if not theta >= 0.0:
        raise ValueError("smoothed aggregation: strength must be >= 0, got %r" % (theta,))
    n = colptr.shape[0] - 1
    d = diagonal(colptr, rowidx, val, level)
    col = np.repeat(np.arange(n), np.diff(colptr))
    thr = theta * np.sqrt(np.abs(d[col]) * np.abs(d[rowidx]))
    return (rowidx != col) & (val != 0.0) & (np.abs(val) > thr)


def aggregate(A, theta=0.08, level=0):
    """(agg, n_aggregates, pass1_roots): agg[i] = aggregate of row i; pass1_roots[J] = root row of a
    pass-1 aggregate J (-1 for the other aggregates)."""
    colptr, rowidx, val = _rows(A)
    n = colptr.shape[0] - 1
    S = strong(colptr, rowidx, val, theta, level)
    nbr = [rowidx[colptr[i]:colptr[i + 1]][S[colptr[i]:colptr[i + 1]]].tolist() for i in range(n)]
    agg = [-1] * n
    roots = []
    for i in range(n):  # pass 1
        if agg[i] < 0 and all(agg[j] < 0 for j in nbr[i]):
            J = len(roots)
            roots.append(i)
            agg[i] = J
            for j in nbr[i]:
                agg[j] = J
    n1 = len(roots)
    in1 = [a >= 0 for a in agg]
    for i in range(n):  # pass 2
        if agg[i] < 0:
            for j in nbr[i]:
                if in1[j]:
                    agg[i] = agg[j]
                    break
    for i in range(n):  # pass 3
        if agg[i] < 0:
            J = len(roots)
            roots.append(-1)
            agg[i] = J
            for j in nbr[i]:
                if agg[j] < 0:
                    agg[j] = J
    roots = np.array(roots, np.int64)
    roots[n1:] = -1
    return np.array(agg, np.int32), len(roots), roots


def prolongation(A, agg, n_agg, level=0):
    """Smoothed P (n x n_agg) as an oracle Csc."""
    colptr, rowidx, val = _rows(A)
    n = colptr.shape[0] - 1
    d = diagonal(colptr, rowidx, val, level)
    col = np.repeat(np.arange(n), np.diff(colptr))
    rowsum = np.zeros(n)
    np.add.at(rowsum, col, np.abs(val))  # unbuffered: ascending stored order per row, from +0
    rho = np.max(rowsum / np.abs(d))
    w = (4.0 / 3.0) / rho
    c = w / d
    key = col.astype(np.int64) * n_agg + agg[rowidx]
    keys, inv = np.unique(key, return_inverse=True)  # ascending (i, J): rows of P in order
    s = np.zeros(keys.shape[0])
    np.add.at(s, inv, val)
    i, J = keys // n_agg, keys % n_agg
    T = (J == agg[i]).astype(np.float64)
    prod = c[i] * s
    p = T - prod
    # rows of P = CSC columns of R = P^T; P = transpose
    rptr = np.zeros(n + 1, np.int64)
    np.add.at(rptr, i + 1, 1)
    rptr = np.cumsum(rptr)
    R = O.Csc.from_arrays(n_agg, n, rptr.astype(np.int32), J.astype(np.int32), p)
    return R.transpose()


def build(A, n_levels, theta=0.08):
    """Level operators and prolongators: (A_list, P_list, R_list, agg_list)."""
    As = [O.Csc.from_arrays(A.rows, A.cols, *_rows(A))]
    Ps, Rs, aggs = [], [], []
    while len(As) < n_levels and As[-1].rows > MAX_COARSE:
        l = len(As) - 1
        agg, n_agg, _ = aggregate(As[-1], theta, l)
        if n_agg >= As[-1].rows:
            if l == 0:
                raise ValueError("smoothed aggregation: the aggregation of level 0 does not reduce it")
            break
        P = prolongation(As[-1], agg, n_agg, l)
        R = P.transpose()
        As.append(O.galerkin(R, As[-1], P))
        Ps.append(P)
        Rs.append(R)
        aggs.append(agg)
    return As, Ps, Rs, aggs


class Multigrid:
    """orc_mg_* (include/amg/multigrid.hpp:151-337) with the smoothed-aggregation transfer; n_levels
    is a cap (self.n_levels: the levels built)."""

    def __init__(self, A, b, n_levels, tolerance=1e-9, every=10, n_iters=100,
                 smoother=O.SMOOTHER_GS, smoother_iters=1, omega=2.0 / 3.0, theta=0.08):
        if every > n_iters:
            raise ValueError("`compute_error_every_n_iters` must be leq to `n_iters`")
        b = np.ascontiguousarray(b, np.float64)
        if A.rows != b.shape[0]:
            raise ValueError("`A` and `b` must have the same number of degrees of freedom")
        self.tolerance, self.every, self.n_iters = tolerance, every, n_iters
        self._A, self._P, self._R, self.aggs = build(A, n_levels, theta)
        self.n_levels = len(self._A)
        self._AT = [a.transpose() for a in self._A]
        self._u = [np.zeros(a.rows) for a in self._A]
        self._f = [b.copy()] + [np.zeros(a.rows) for a in self._A[1:]]
        self._color = [None] * self.n_levels
        self.coarse = O.Ldlt(self._A[-1])
        self.set_smoother(smoother, smoother_iters, omega)
        self.iters_done, self.last_error, self.hist = 0, 100.0, []

    def set_smoother(self, smoother, smoother_iters=1, omega=2.0 / 3.0):
        self.smoother, self.smoother_iters, self.omega = smoother, smoother_iters, omega
        if smoother == O.SMOOTHER_COLOR_GS:
            for l in range(self.n_levels):
                if self._color[l] is None:
                    self._color[l] = O.greedy_coloring(self._A[l], self._AT[l])

    def n_dofs(self, l):
        return self._A[l].rows

    def A(self, l):
        return self._A[l]

    def P(self, l):
        return self._P[l]

    def R(self, l):
        return self._R[l]

    def u(self, l):
        return self._u[l]

    def f(self, l):
        return self._f[l]

    def operator_complexity(self):
        return sum(a.nnz for a in self._A) / self._A[0].nnz

    def reset(self):
        for u in self._u:
            u[:] = 0.0

    def smooth(self, l):  # orc_mg_smooth
        u, f = self._u[l], self._f[l]
        if self.smoother == O.SMOOTHER_GS:
            O.gs_smooth(self._A[l], u, f, 1e-9, 0, self.smoother_iters)
        elif self.smoother == O.SMOOTHER_JACOBI:
            for _ in range(self.smoother_iters):
                u[:] = O.jacobi_sweep(self._AT[l], u, f, self.omega)
        else:
            nc, color = self._color[l]
            for _ in range(self.smoother_iters):
                for c in list(range(nc)) + list(range(nc - 1, -1, -1)):
                    O.color_gs_pass(self._AT[l], color, c, f, u)

    def vcycle(self):  # orc_mg_vcycle
        L = self.n_levels
        for l in range(L):
            self.smooth(l)
            if l + 1 != L:
                r = O.residual(self._A[l], self._u[l], self._f[l])
                self._u[l + 1][:] = 0.0
                self._f[l + 1][:] = O.spmv(self._R[l], r)
        self._u[L - 1][:] = self.coarse.solve(self._f[L - 1])
        for l in range(L - 2, -1, -1):
            self._u[l][:] = self._u[l] + O.spmv(self._P[l], self._u[l + 1])
            self.smooth(l)

    def rss(self):
        return O.rss(self._A[0], self._u[0], self._f[0])

    def solve(self):  # orc_mg_solve
        it, error, self.hist = 0, 100.0, []
        while it < self.n_iters and error > self.tolerance:
            self.vcycle()
            it += 1
            if self.every != 0 and it % self.every == 0:
                error = self.rss()
                self.hist.append(error)
        self.iters_done, self.last_error = it, error
        return it

    def solve_relative(self, rel_tol):
        """Cycles until ||b - A u|| / ||b|| <= rel_tol (checked every `every` cycles), capped at n_iters."""
        bnorm2 = float(np.dot(self._f[0], self._f[0]))
        it, rel = 0, np.inf
        every = max(1, self.every)
        while it < self.n_iters and rel > rel_tol:
            self.vcycle()
            it += 1
            if it % every == 0:
                rel = (self.rss() / bnorm2) ** 0.5
        self.iters_done, self.last_error = it, rel
        return it

    def precondition(self, r):
        """z = one V-cycle on A z = r from z = 0 (the level-0 state is overwritten)."""
        return precondition(self, r)

    def solve_pcg(self, b, rel_tol, max_iters=1000):
        """Iterations of amgb_solve_pcg's recurrences (numpy dot products) to rel_tol from u = 0; the
        level-0 state ends as (b, x)."""
        it, rel, x = pcg(self._A[0], b, lambda r: precondition(self, r), rel_tol, max_iters)
        self._f[0][:] = b
        self._u[0][:] = x
        self.iters_done, self.last_error = it, rel
        return it


def precondition(mg, r):
    """z = one V-cycle of multigrid `mg` (this module's or the oracle's) on A z = r from z = 0."""
    mg.f(0)[:] = r
    mg.u(0)[:] = 0.0
    mg.vcycle()
    return mg.u(0).copy()


def pcg(A, b, prec, rel_tol, max_iters=1000):
    """amgb_solve_pcg in numpy: conjugate gradients on A x = b from x = 0, preconditioned by prec(r);
    returns (iterations, ||r|| / ||b||, x)."""
    b = np.ascontiguousarray(b, np.float64)
    x = np.zeros_like(b)
    r = b.copy()
    bnorm2 = float(np.dot(b, b))
    rel = np.sqrt(float(np.dot(r, r)) / bnorm2)
    zero = np.zeros_like(b)
    p, rz_old, it = None, 0.0, 0
    while it < max_iters and rel > rel_tol:
        z = prec(r)
        rz = float(np.dot(r, z))
        p = z.copy() if it == 0 else z + (rz / rz_old) * p
        q = O.residual(A, p, zero)  # -A p
        pq = float(np.dot(p, q))
        if pq == 0.0 or not np.isfinite(pq):
            break
        alpha = -rz / pq
        x = x + alpha * p
        r = r + alpha * q
        rz_old = rz
        rel = np.sqrt(float(np.dot(r, r)) / bnorm2)
        it += 1
    return it, rel, x


# ---- test matrices (CSC triples with ascending row indices) ----
def _csc(M):
    import scipy.sparse as sp
    M = sp.csc_matrix(M)
    M.sort_indices()
    return O.Csc.from_arrays(M.shape[0], M.shape[1], M.indptr, M.indices, M.data)


def rectangular_poisson(nx, ny):
    """5-point Poisson on an nx x ny grid (x fastest), built with scipy kron."""
    import scipy.sparse as sp

    def t(n):
        return sp.diags([np.ones(n - 1), -2.0 * np.ones(n), np.ones(n - 1)], [-1, 0, 1]) * float((n + 1) ** 2)
    return _csc(sp.kron(sp.identity(ny), t(nx)) + sp.kron(t(ny), sp.identity(nx)))


def permuted_laplacian(m, seed=0):
    """Grid::laplacian(m) with rows and columns renumbered by a seeded random permutation; returns
    (A, perm) with A = Q L Q^T, row k of A = row perm[k] of L."""
    L = O.laplacian(m).to_scipy()
    perm = np.random.default_rng(seed).permutation(m * m)
    return _csc(L[perm][:, perm]), perm


def lognormal_diffusion(m, sigma=1.0, seed=0):
    """-div(k grad u) on an m x m grid, 5-point, with seeded lognormal edge coefficients (Dirichlet
    boundary edges included): A = sum_e k_e (e_i - e_j)(e_i - e_j)^T + boundary terms, negated so that
    its sign matches Grid::laplacian."""
    import scipy.sparse as sp
    rng = np.random.default_rng(seed)
    idx = np.arange(m * m).reshape(m, m)
    rows, cols, vals = [], [], []
    diag = np.zeros(m * m)
    for a, b in ((idx[:, :-1], idx[:, 1:]), (idx[:-1, :], idx[1:, :])):
        a, b = a.ravel(), b.ravel()
        k = np.exp(sigma * rng.standard_normal(a.size))
        rows += [a, b]
        cols += [b, a]
        vals += [-k, -k]
        np.add.at(diag, a, k)
        np.add.at(diag, b, k)
    for border in (idx[0, :], idx[-1, :], idx[:, 0], idx[:, -1]):
        np.add.at(diag, border, np.exp(sigma * rng.standard_normal(border.size)))
    rows.append(idx.ravel())
    cols.append(idx.ravel())
    vals.append(diag)
    M = sp.coo_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))), shape=(m * m, m * m))
    return _csc(-M.tocsc() * float((m + 1) ** 2))
