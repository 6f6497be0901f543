// Galerkin coarse operator A_H = R (A P) for the bilinear transfer (AMGB_TRANSFER_BILINEAR_2D),
// evaluated row by row on the DIA layout: the device-side setup of 2-D hierarchies.
//
// The fine operator lives on an m_h x m_h grid (DOF k = y*m_h + x) and couples every point only to
// its 3 x 3 neighbourhood (offsets in {+-m_h+-1, +-m_h, +-1, 0}, no entry across a line end).  P =
// P1 (x) P1 with P1 = LinearInterpolator's pattern, m_H = m_h / 2, R = P^T.  Column J = (Y, X) of
// P holds the fine points (2Y + a, 2X + b), a, b in {0, 1, 2}, inside the grid, with weight
// w(a) * w(b), w = (.5, 1, .5).  The coarse operator is again a 3 x 3 grid stencil: nine coarse
// diagonals {+-m_H+-1, +-m_H, +-1, 0}.
//
// Eigen's conservative product evaluates T = A P first -- T(i, J) accumulates A(i, k) P(k, J) over
// ascending k -- and then R T -- A_H(I, J) accumulates R(I, i) T(i, J) over ascending i.
// coarse_entry_2d keeps exactly that order (ascending k is y-major over the 3 x 3 support), so its
// values are bit-identical to host_setup.cpp's galerkin() with make_prolongation_2d for every entry.
// Absent entries and explicit zeros contribute +0 in either formulation.
#pragma once

#include "galerkin_dia.cuh"

namespace amgb {
namespace gal {

constexpr int kCoarseDiag2d = 9;

// The distinct coarse offsets dy * m_H + dx (dy, dx in {-1, 0, 1}), ascending; returns their number
// (nine for m_H >= 3, fewer on the smallest grids where some coincide).
AMGB_GAL_FN int coarse_offsets_2d(int m_H, int* off_c) {
  int n = 0;
  for (int dy = -1; dy <= 1; ++dy)
    for (int dx = -1; dx <= 1; ++dx) {
      const int o = dy * m_H + dx;
      int p = n;
      while (p > 0 && off_c[p - 1] > o) --p;
      if (p > 0 && off_c[p - 1] == o) continue;
      for (int q = n; q > p; --q) off_c[q] = off_c[q - 1];
      off_c[p] = o;
      ++n;
    }
  return n;
}

// A_H(I, J) in Eigen's evaluation order (A.n == m_h * m_h).
AMGB_GAL_FN double coarse_entry_2d(const FineDia& A, int m_h, int m_H, int I, int J) {
  const int n_c = m_H * m_H;
  if (I < 0 || I >= n_c || J < 0 || J >= n_c) return 0.0;
  const int YI = I / m_H, XI = I - YI * m_H, YJ = J / m_H, XJ = J - YJ * m_H;
  double acc = 0.0;
  for (int ai = 0; ai < 3; ++ai) {  // R(I, i) = P(i, I), ascending i
    const int yi = 2 * YI + ai;
    if (yi >= m_h) break;
    const double wyi = (ai == 1) ? 1.0 : 0.5;
    for (int bi = 0; bi < 3; ++bi) {
      const int xi = 2 * XI + bi;
      if (xi >= m_h) break;
      const double wi = wyi * ((bi == 1) ? 1.0 : 0.5);  // exact: powers of two
      const int i = yi * m_h + xi;
      double t = 0.0;  // T(i, J) = sum over ascending k of A(i, k) P(k, J)
      for (int ak = 0; ak < 3; ++ak) {
        const int yk = 2 * YJ + ak;
        if (yk >= m_h) break;
        const double wyk = (ak == 1) ? 1.0 : 0.5;
        for (int bk = 0; bk < 3; ++bk) {
          const int xk = 2 * XJ + bk;
          if (xk >= m_h) break;
          const double a = fine_entry(A, i, yk * m_h + xk);
          if (a != 0.0) t = gadd(t, gmul(a, wyk * ((bk == 1) ? 1.0 : 0.5)));
        }
      }
      if (t != 0.0) acc = gadd(acc, gmul(wi, t));
    }
  }
  return acc;
}

// One coarse row: out[c * out_stride] = A_H(I, I + off_c[c]) for the nd_c offsets of coarse_offsets_2d.
AMGB_GAL_FN void coarse_row_2d(const FineDia& A, int m_h, int m_H, int nd_c, const int* off_c, int I, double* out,
                               int out_stride) {
  for (int c = 0; c < nd_c; ++c) out[(long long)c * out_stride] = coarse_entry_2d(A, m_h, m_H, I, I + off_c[c]);
}

}  // namespace gal
}  // namespace amgb
