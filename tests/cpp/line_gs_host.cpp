// TEST INFRASTRUCTURE ONLY -- never linked into libamgb.so.
// Host build of algebraic-multigrid_b200/csrc/line_gs.cuh (zebra line Gauss-Seidel) for
// tests/test_linegs2d_host.py: the setup factors and one pass, in the kernels' data layout (t and the
// factors step-major, the forward sweep in place over t) and with their per-row functions.
#include "../../algebraic-multigrid_b200/csrc/line_gs.cuh"

namespace {
amgb::lgs::Grid grid(int m, int nd, const int* off, int ld, const double* val, int* ok) {
  const amgb::gsw::Plan P = amgb::gsw::plan_for(off, nd, m * m, m);
  *ok = P.ok ? 1 : 0;
  amgb::lgs::Grid G{};
  G.val = val;
  G.ld = ld;
  G.m = m;
  for (int e = 0; e < amgb::gsw::kSlots; ++e) G.d_of[e] = P.ok ? P.d_of[e] : -1;
  return G;
}
}  // namespace

extern "C" {

// Rows of A in DIA (nd ascending offsets, val[d * ld + k]).  Writes sub / den / cp (n doubles each,
// step-major: index p * m + line) of direction D (0: X, 1: Y).  Returns -2 when the offsets do not
// decode as a 3 x 3 grid stencil, else the first zero-pivot row or -1.
int lgs_host_factor(int m, int D, int nd, const int* off, int ld, const double* val, double* sub, double* den,
                    double* cp) {
  int ok = 0;
  const amgb::lgs::Grid G = grid(m, nd, off, ld, val, &ok);
  if (!ok) return -2;
  int bad = -1;
  for (int line = 0; line < m; ++line) {
    const int k = amgb::lgs::factor_line<false>(G, D, line, sub, den, cp);
    if (k >= 0 && (bad < 0 || k < bad)) bad = k;
  }
  return bad;
}

// One pass over the lines of direction D and colour c, u updated in place (g: n scratch doubles).
int lgs_host_pass(int m, int D, int c, int nd, const int* off, int ld, const double* val, const double* sub,
                  const double* den, const double* cp, const double* f, double* u, double* g) {
  using namespace amgb::lgs;
  int ok = 0;
  const Grid G = grid(m, nd, off, ld, val, &ok);
  if (!ok) return -2;
  for (int line = c; line < m; line += 2)
    for (int p = 0; p < m; ++p) {
      const int k = row_of(D, m, line, p);
      g[smj(m, line, p)] = D == kX ? line_rhs<kX, false>(G, f, u, k) : line_rhs<kY, false>(G, f, u, k);
    }
  for (int line = c; line < m; line += 2) {
    double prev = 0.0;
    for (int p = 0; p < m; ++p) {
      const int i = smj(m, line, p);
      prev = fwd_step<false>(g[i], sub[i], den[i], prev, p == 0);
      g[i] = prev;
    }
    for (int p = m - 1; p >= 0; --p) {
      const int i = smj(m, line, p);
      prev = bwd_step<false>(g[i], cp[i], prev, p == m - 1);
      u[row_of(D, m, line, p)] = prev;
    }
  }
  return 0;
}
}
