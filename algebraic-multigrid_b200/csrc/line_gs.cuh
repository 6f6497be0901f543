// Zebra line Gauss-Seidel on the levels of a 2-D hierarchy (AMGB_SMOOTHER_LINE_GS).
//
// A level is an m x m grid operator with k = y*m + x whose entries couple (y, x) only with
// (y + a, x + d), |a|, |d| <= 1, never across the end of a line (the k_gsw_check criterion).  An
// X-line is the m rows of one y (neighbours along it at +-1), a Y-line the m rows of one x
// (neighbours at +-m); a line's colour is its index mod 2.  A pass over direction D and colour c
// solves, for every line of colour c,
//   t_i = f_i - sum_{j not on the line} a_ij u_j   (non-zero stored entries, ascending j, separate
//                                                  multiply and subtract)
//   T u_line = t                                   (T: the line's tridiagonal block, Thomas)
// with the factors of setup time
//   den_0 = a_00,  den_p = a_pp - a_{p,p-1} cp_{p-1},  cp_p = a_{p,p+1} / den_p
// and the sweeps
//   y_0 = t_0 / den_0,  y_p = (t_p - a_{p,p-1} y_{p-1}) / den_p;  u_{m-1} = y_{m-1},  u_p = y_p - cp_p u_{p+1}.
// Lines of one colour read only lines of the other colour, so a pass does not depend on the order
// in which its lines run.  The reference arithmetic is exactly these operations (IEEE division, no
// FMA): bit-identical to tests/oracle_linegs2d.py.  FAST stores 1 / den and contracts to FMAs.
//
// Layout.  Every line runs one sequential recurrence (no segment-parallel solve: it would change the
// rounding).  A pass is two launches: k_line_rhs computes t for all rows of the colour at once (one
// thread per row, coalesced reads of A, f and u) and writes it to a scratch vector g in STEP-MAJOR
// order, g[p * m + line]; k_line_solve runs one thread per line over p and reads g and the factors,
// stored in the same step-major order, so the 32 lanes of a warp (lines line0 + 2j) read addresses 16
// bytes apart.  For Y-lines step-major is the natural order; for X-lines it is the transposed grid.
// The forward sweep writes y over t in g, the backward sweep writes u in natural order.
#pragma once
#include <climits>
#include <cmath>

#include "gs_wave.cuh"

#if defined(__CUDACC__)
#define LGS_HD __host__ __device__ __forceinline__
#else
#define LGS_HD inline
#endif

namespace amgb {
namespace lgs {

constexpr int kX = 0;  // X-lines: the rows of one y
constexpr int kY = 1;  // Y-lines: the rows of one x
constexpr int kSolveThreads = 32;
constexpr int kBatch = 8;  // steps whose loads are issued together in k_line_solve

// the level in DIA form (rows of A, val[d * ld + k], 0.0 = no entry) and the diagonal of each
// stencil slot e = (a + 1) * 3 + (d + 1) (-1: absent); slots ascend with the memory offset a*m + d
struct Grid {
  const double* val;
  int ld;
  int m;
  int d_of[gsw::kSlots];
};

// slots of the tridiagonal block along direction D: below, diagonal, above
LGS_HD int slot_sub(int D) { return D == kX ? 3 : 1; }
LGS_HD int slot_sup(int D) { return D == kX ? 5 : 7; }
// the six slots off the line, ascending memory offset
LGS_HD int off_slot(int D, int i) {
  // X: (-1,-1) (-1,0) (-1,1) (1,-1) (1,0) (1,1);  Y: (-1,-1) (-1,1) (0,-1) (0,1) (1,-1) (1,1)
  return D == kX ? (i < 3 ? i : i + 3) : (i < 2 ? 2 * i : (i < 4 ? 2 * i - 1 : 2 * i - 2));
}
LGS_HD int slot_offset(int m, int e) { return (e / 3 - 1) * m + (e % 3 - 1); }
LGS_HD double coef(const Grid& G, int e, int k) {
  const int d = G.d_of[e];
  return d < 0 ? 0.0 : G.val[(size_t)d * (size_t)G.ld + (size_t)k];
}
// natural index of step p of line `line`, and its step-major index
LGS_HD int row_of(int D, int m, int line, int p) { return D == kX ? line * m + p : p * m + line; }
LGS_HD int smj(int m, int line, int p) { return p * m + line; }

LGS_HD double fms(double a, double b, double c, bool fast) {  // c - a * b
#if defined(__CUDA_ARCH__)
  return fast ? __fma_rn(-a, b, c) : __dsub_rn(c, __dmul_rn(a, b));
#else
  return fast ? std::fma(-a, b, c) : c - a * b;
#endif
}

// t of row k on a line of direction D
template <int D, bool FAST>
LGS_HD double line_rhs(const Grid& G, const double* f, const double* u, int k) {
  double t = f[k];
#pragma unroll
  for (int i = 0; i < 6; ++i) {
    const int e = off_slot(D, i);
    const double c = coef(G, e, k);
    if (c != 0.0) t = fms(c, u[k + slot_offset(G.m, e)], t, FAST);
  }
  return t;
}

// Factors of one line (setup): sub[], den[] (FAST: 1 / den), cp[] at the step-major indices.
// Returns the natural index of the first zero pivot, or -1.
template <bool FAST>
LGS_HD int factor_line(const Grid& G, int D, int line, double* sub, double* den, double* cp) {
  const int m = G.m;
  double cprev = 0.0;
  for (int p = 0; p < m; ++p) {
    const int k = row_of(D, m, line, p);
    const double s = coef(G, slot_sub(D), k);
    const double a = coef(G, 4, k);
    const double dn = p == 0 ? a : gsw::sub_(a, gsw::mul_(s, cprev));
    if (dn == 0.0) return k;
    cprev = gsw::div_(coef(G, slot_sup(D), k), dn);
    const int q = smj(m, line, p);
    sub[q] = s;
    den[q] = FAST ? gsw::div_(1.0, dn) : dn;
    cp[q] = cprev;
  }
  return -1;
}

// one forward / backward step of the Thomas sweeps
template <bool FAST>
LGS_HD double fwd_step(double t, double s, double dn, double yprev, bool first) {
  const double num = first ? t : fms(s, yprev, t, FAST);
  return FAST ? gsw::mul_(num, dn) : gsw::div_(num, dn);
}
template <bool FAST>
LGS_HD double bwd_step(double y, double c, double unext, bool last) {
  return last ? y : fms(c, unext, y, FAST);
}

// lines of colour c: c, c + 2, ...
LGS_HD int lines_of_colour(int m, int c) { return (m - c + 1) / 2; }

#if defined(__CUDACC__)
// one thread per line of direction D (all m lines); *bad = smallest natural row with a zero pivot
template <bool FAST>
__global__ void __launch_bounds__(128) k_line_factor(Grid G, int D, double* sub, double* den, double* cp, int* bad) {
  const int line = blockIdx.x * blockDim.x + threadIdx.x;
  if (line >= G.m) return;
  const int k = factor_line<FAST>(G, D, line, sub, den, cp);
  if (k >= 0) atomicMin(bad, k);
}

// t of every row on the lines of colour c, written step-major to g
template <int D, bool FAST>
__global__ void __launch_bounds__(256) k_line_rhs(Grid G, int c, const double* __restrict__ f,
                                                  const double* __restrict__ u, double* __restrict__ g) {
  const int m = G.m;
  const int nl = lines_of_colour(m, c);
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nl * m) return;
  int line, p;
  if (D == kX) {  // consecutive threads walk along a line: contiguous rows
    line = c + 2 * (i / m);
    p = i % m;
  } else {  // consecutive threads take consecutive lines of the colour within one row y = p
    line = c + 2 * (i % nl);
    p = i / nl;
  }
  g[smj(m, line, p)] = line_rhs<D, FAST>(G, f, u, row_of(D, m, line, p));
}

// the two Thomas sweeps of every line of colour c: lane j of the grid owns line c + 2 j
template <int D, bool FAST>
__global__ void __launch_bounds__(kSolveThreads) k_line_solve(int m, int c, const double* __restrict__ sub,
                                                               const double* __restrict__ den,
                                                               const double* __restrict__ cp, double* g,
                                                               double* u) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= lines_of_colour(m, c)) return;
  const int line = c + 2 * j;
  double prev = 0.0;
  for (int p0 = 0; p0 < m; p0 += kBatch) {
    double t[kBatch], s[kBatch], dn[kBatch];
#pragma unroll
    for (int q = 0; q < kBatch; ++q)
      if (p0 + q < m) {
        const int i = smj(m, line, p0 + q);
        t[q] = g[i];
        s[q] = sub[i];
        dn[q] = den[i];
      }
#pragma unroll
    for (int q = 0; q < kBatch; ++q)
      if (p0 + q < m) {
        prev = fwd_step<FAST>(t[q], s[q], dn[q], prev, p0 + q == 0);
        t[q] = prev;
      }
#pragma unroll
    for (int q = 0; q < kBatch; ++q)
      if (p0 + q < m) g[smj(m, line, p0 + q)] = t[q];
  }
  const int top = (m - 1) / kBatch * kBatch;  // batches in reverse, aligned like the forward ones
  for (int p0 = top; p0 >= 0; p0 -= kBatch) {
    double y[kBatch], cc[kBatch];
#pragma unroll
    for (int q = kBatch - 1; q >= 0; --q)
      if (p0 + q < m) {
        const int i = smj(m, line, p0 + q);
        y[q] = g[i];
        cc[q] = cp[i];
      }
#pragma unroll
    for (int q = kBatch - 1; q >= 0; --q)
      if (p0 + q < m) {
        prev = bwd_step<FAST>(y[q], cc[q], prev, p0 + q == m - 1);
        y[q] = prev;
      }
#pragma unroll
    for (int q = kBatch - 1; q >= 0; --q)
      if (p0 + q < m) u[row_of(D, m, line, p0 + q)] = y[q];
  }
}
#endif

}  // namespace lgs
}  // namespace amgb
