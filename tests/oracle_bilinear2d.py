"""CPU oracle of the bilinear 2-D transfer (TRANSFER_BILINEAR_2D).  TEST INFRASTRUCTURE ONLY.

The transfer has no reference counterpart: this definition is the specification.  It is built
from the CPU oracle's own operations (oracle/amg_oracle.c: the 1-D P of LinearInterpolator, the
transpose, Eigen's conservative product order, the residual, spmv, the three smoothers and the
banded LDL^T), composed exactly like orc_mg_create / orc_mg_vcycle / orc_mg_solve compose them;
only P differs:
  - grid of m x m DOFs numbered k = y*m + x (the numbering of Grid::laplacian);
  - m_H = m_h // 2 (every fine line is covered by a coarse line also when m_h is even);
  - P = P1 (x) P1, P1 = oracle.make_P(m_h, m_H): column (Y, X) holds rows (y, x) for y in column Y
    and x in column X of P1, y-major (ascending row), value P1(y, Y) * P1(x, X) (exact: powers of 2);
  - R = P^T (no 1/4 scaling), A_H = R (A P).
"""
import numpy as np

import oracle as O


def coarse_lines(m_h):
    return m_h // 2


def make_P2d(m_h, m_H):
    """P = P1 (x) P1 as an oracle CSC matrix (m_h^2 x m_H^2)."""
    c1, r1, v1 = O.make_P(m_h, m_H).arrays()
    cnt1 = np.diff(c1).astype(np.int64)            # rows per column of P1 (3, or 2 in the last column)
    cnt = np.outer(cnt1, cnt1).reshape(-1)          # column (Y, X) holds cnt1[Y] * cnt1[X] rows
    colptr = np.concatenate([[0], np.cumsum(cnt)]).astype(np.int32)
    # slot s of column (Y, X): y = s // cnt1[X] -th row of column Y, x = s % cnt1[X] -th row of column X
    col = np.repeat(np.arange(m_H * m_H, dtype=np.int64), cnt)
    s = np.arange(int(cnt.sum()), dtype=np.int64) - np.repeat(colptr[:-1].astype(np.int64), cnt)
    Y, X = col // max(m_H, 1), col % max(m_H, 1)
    py = c1[Y] + s // cnt1[X]
    px = c1[X] + s % cnt1[X]
    rowidx = (r1[py].astype(np.int64) * m_h + r1[px]).astype(np.int32)
    val = v1[py] * v1[px]
    return O.Csc.from_arrays(m_h * m_h, m_H * m_H, colptr, rowidx, val)


def level_sizes(m0, n_levels):
    m = [m0]
    for _ in range(1, n_levels):
        m.append(coarse_lines(m[-1]))
    return [k * k for k in m]


class Multigrid:
    """orc_mg_* (include/amg/multigrid.hpp:151-337) with the bilinear 2-D transfer."""

    def __init__(self, A, b, n_levels, tolerance=1e-9, every=10, n_iters=100,
                 smoother=O.SMOOTHER_GS, smoother_iters=1, omega=2.0 / 3.0):
        if every > n_iters:
            raise ValueError("`compute_error_every_n_iters` must be leq to `n_iters`")
        b = np.ascontiguousarray(b, np.float64)
        if A.rows != b.shape[0]:
            raise ValueError("`A` and `b` must have the same number of degrees of freedom")
        m0 = int(round(A.rows ** 0.5))
        if m0 * m0 != A.rows:
            raise ValueError("the bilinear 2-D transfer needs an m x m grid operator")
        self.n_levels, self.tolerance, self.every, self.n_iters = n_levels, tolerance, every, n_iters
        self.m = [m0]
        self._A, self._P, self._R = [O.Csc.from_arrays(A.rows, A.cols, *A.arrays())], [], []
        for l in range(1, n_levels):
            m_H = coarse_lines(self.m[-1])
            if m_H < 1:
                raise ValueError("too many levels: level %d is empty" % l)
            self._P.append(make_P2d(self.m[-1], m_H))
            self._R.append(self._P[-1].transpose())
            self._A.append(O.galerkin(self._R[-1], self._A[-1], self._P[-1]))
            self.m.append(m_H)
        self._AT = [a.transpose() for a in self._A]
        self._u = [np.zeros(k * k) for k in self.m]
        self._f = [b.copy()] + [np.zeros(k * k) for k in self.m[1:]]
        self._color = [None] * n_levels
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
        return self.m[l] * self.m[l]

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
