"""CPU oracle of zebra line Gauss-Seidel (SMOOTHER_LINE_GS) on 2-D hierarchies.  TEST INFRASTRUCTURE ONLY.

The smoother has no reference counterpart: this definition is the specification (include/amgb.h,
AMGB_SMOOTHER_LINE_GS).  Levels are m x m grids, k = y*m + x.  An X-line is the m rows of one y, a
Y-line the m rows of one x; a line's colour is its index mod 2.  A pass over direction D and colour c,
for every line of colour c:
  t_i = f_i - a_ij u_j over the non-zero stored entries of row i of A off the line, ascending j
        (separate multiply and subtract);
  Thomas along the line: den_0 = a_00, cp_p = a_{p,p+1} / den_p, den_p = a_pp - a_{p,p-1} cp_{p-1};
        y_0 = t_0 / den_0, y_p = (t_p - a_{p,p-1} y_{p-1}) / den_p; u_{m-1} = y_{m-1},
        u_p = y_p - cp_p u_{p+1}.
One iteration = forward half (directions in order, colour 0 then 1) + backward half (directions
reversed, colour 1 then 0).  numpy's element-wise float64 operations are single IEEE operations, so the
code below, vectorised across the lines of a colour and sequential along them, is that order exactly.
"""
import numpy as np

import oracle as O
import oracle_bilinear2d as O2

SMOOTHER_LINE_GS = 3
LINES_X, LINES_Y, LINES_ALTERNATING = 0, 1, 2
X, Y = 0, 1
DIRS = {LINES_X: (X,), LINES_Y: (Y,), LINES_ALTERNATING: (X, Y)}
# stencil slot e = (a + 1) * 3 + (d + 1) couples (y, x) with (y + a, x + d); ascending e = ascending j
SUB, SUP = {X: 3, Y: 1}, {X: 5, Y: 7}
OFF_LINE = {X: (0, 1, 2, 6, 7, 8), Y: (0, 2, 3, 5, 6, 8)}


def slots(A, m):
    """C[e, k] = A(k, k + offset of slot e) for the rows of A (0.0 = no entry); ValueError when an entry
    is not a 3 x 3 grid neighbour (or couples across the end of a line)."""
    n = m * m
    c, r, v = A.transpose().arrays()  # column k of A^T = row k of A
    k = np.repeat(np.arange(n), np.diff(c))
    j = r.astype(np.int64)
    dy, dx = j // m - k // m, j % m - k % m
    live = v != 0.0
    if np.any(live & ((np.abs(dy) > 1) | (np.abs(dx) > 1))):
        raise ValueError("not an m x m grid operator with a 3 x 3 stencil")
    C = np.zeros((9, n))
    C[((dy + 1) * 3 + dx + 1)[live], k[live]] = v[live]
    return C


def lines_view(a, m, D):
    """[line, p] view of a natural-order vector of n = m*m entries along direction D."""
    g = a.reshape(m, m)  # [y, x]
    return g if D == X else g.T


def slot_offset(m, e):
    return (e // 3 - 1) * m + (e % 3 - 1)


def factors(C, m, D):
    """sub, den, cp as [line, p] arrays; ValueError naming the natural row of a zero pivot."""
    sub = lines_view(C[SUB[D]], m, D)
    dia = lines_view(C[4], m, D)
    sup = lines_view(C[SUP[D]], m, D)
    den, cp = np.zeros((m, m)), np.zeros((m, m))
    for p in range(m):
        den[:, p] = dia[:, p] if p == 0 else dia[:, p] - sub[:, p] * cp[:, p - 1]
        if np.any(den[:, p] == 0.0):
            line = int(np.nonzero(den[:, p] == 0.0)[0][0])
            raise ValueError("zero pivot at row %d" % (line * m + p if D == X else p * m + line))
        cp[:, p] = sup[:, p] / den[:, p]
    return sub.copy(), den, cp


def line_rhs(C, m, D, f, u):
    """t of every row (natural order); only the rows of the lines being solved are used."""
    n = m * m
    k = np.arange(n)
    t = f.copy()
    for e in OFF_LINE[D]:
        c = C[e]
        nb = u[np.clip(k + slot_offset(m, e), 0, n - 1)]
        t = np.where(c != 0.0, t - c * nb, t)
    return t


def thomas(t, sub, den, cp):
    """Rows of t ([lines, p]) solved with the factors of the same lines."""
    nl, m = t.shape
    y = np.zeros((nl, m))
    for p in range(m):
        y[:, p] = t[:, p] / den[:, p] if p == 0 else (t[:, p] - sub[:, p] * y[:, p - 1]) / den[:, p]
    u = np.zeros((nl, m))
    u[:, m - 1] = y[:, m - 1]
    for p in range(m - 2, -1, -1):
        u[:, p] = y[:, p] - cp[:, p] * u[:, p + 1]
    return u


def line_pass(C, fac, m, D, c, f, u):
    """One pass over the lines of direction D and colour c; u (natural order) is updated in place."""
    sub, den, cp = fac
    t = lines_view(line_rhs(C, m, D, f, u), m, D)
    L = np.arange(c, m, 2)
    lines_view(u, m, D)[L] = thomas(t[L], sub[L], den[L], cp[L])


class LineSmoother:
    """The smoother on one m x m grid operator (the SmootherBase::smooth boundary)."""

    def __init__(self, A, lines=LINES_X):
        m = int(round(A.rows ** 0.5))
        if m * m != A.rows:
            raise ValueError("line Gauss-Seidel needs an m x m grid operator")
        self.m, self.dirs = m, DIRS[lines]
        self.C = slots(A, m)
        self.fac = {D: factors(self.C, m, D) for D in self.dirs}

    def half(self, f, u, forward):
        for D in (self.dirs if forward else self.dirs[::-1]):
            for c in ((0, 1) if forward else (1, 0)):
                line_pass(self.C, self.fac[D], self.m, D, c, f, u)

    def smooth(self, f, u, n_iters=1):
        for _ in range(n_iters):
            self.half(f, u, True)
            self.half(f, u, False)


class Multigrid(O2.Multigrid):
    """oracle_bilinear2d.Multigrid with SMOOTHER_LINE_GS (lines: LINES_*)."""

    def __init__(self, A, b, n_levels, tolerance=1e-9, every=10, n_iters=100,
                 smoother=SMOOTHER_LINE_GS, smoother_iters=1, omega=2.0 / 3.0, lines=LINES_X):
        self.lines = lines
        self._line = None
        super().__init__(A, b, n_levels, tolerance, every, n_iters, smoother, smoother_iters, omega)

    def set_smoother(self, smoother, smoother_iters=1, omega=2.0 / 3.0):
        if smoother != SMOOTHER_LINE_GS:
            return super().set_smoother(smoother, smoother_iters, omega)
        self.smoother, self.smoother_iters, self.omega = smoother, smoother_iters, omega
        if self._line is None:
            self._line = [LineSmoother(self._A[l], self.lines) for l in range(self.n_levels)]

    def smooth(self, l):
        if self.smoother != SMOOTHER_LINE_GS:
            return super().smooth(l)
        self._line[l].smooth(self._f[l], self._u[l], self.smoother_iters)
