// TEST INFRASTRUCTURE ONLY -- never linked into libamgb.so.
// Host build of algebraic-multigrid_b200/csrc/galerkin_dia2d.cuh (the row-wise Galerkin product of the
// bilinear 2-D transfer on the DIA layout, the device-side setup of 2-D hierarchies) for
// tests/test_bilinear2d_host.py.
#include "../../algebraic-multigrid_b200/csrc/galerkin_dia2d.cuh"

extern "C" {

// Fine operator on an m_h x m_h grid: nd_f ascending offsets, val_f[d * ld_f + row].  Writes the
// coarse offsets to off_c (capacity 9), their number to *nd_c and the values of the m_H x m_H
// coarse operator to val_c[c * ld_c + I].
void gal2d_host_coarse(int m_h, int nd_f, const int* off_f, int ld_f, const double* val_f, int m_H, int* off_c,
                       int* nd_c, int ld_c, double* val_c) {
  amgb::gal::FineDia A;
  A.n = m_h * m_h;
  A.nd = nd_f;
  A.ld = ld_f;
  for (int d = 0; d < nd_f; ++d) A.off[d] = off_f[d];
  A.val = val_f;
  const int n = amgb::gal::coarse_offsets_2d(m_H, off_c);
  *nd_c = n;
  for (int I = 0; I < m_H * m_H; ++I) amgb::gal::coarse_row_2d(A, m_h, m_H, n, off_c, I, val_c + I, ld_c);
}
}
