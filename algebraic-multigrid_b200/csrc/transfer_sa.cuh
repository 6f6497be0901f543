// Grid transfers of a smoothed-aggregation hierarchy (AMGB_TRANSFER_SMOOTHED_AGGREGATION, sm_100a).
// P is an arbitrary sparse matrix, so both transfers are SELL-32 row walks, one thread per output row:
//   k_restrict_sa     f_c = R r with R = P^T: the view holds the rows of R (the CSC columns of P);
//                     also zeroes u_c (multigrid.hpp:278-282)
//   k_prolong_add_sa  u = u + (P e): the view holds the rows of P; P e is accumulated from +0 and
//                     added once, as the oracle's u + spmv(P, e) does (multigrid.hpp:294-296)
// Every row walks its entries in ascending column order, which is the order in which Eigen's sparse x
// dense product (the oracle's spmv) accumulates them.  The residual that the restriction reads is formed
// beforehand by k_residual: rows of R overlap, so fusing it in would form each residual several times.
// FAST = false: separate __dmul_rn / __dadd_rn, bit-identical to tests/oracle_sa.py (the weights of a
// smoothed P are not powers of two, so a contraction would change the bits).  FAST = true: FMAs.
#pragma once
#include "kernels.cuh"

namespace amgb {
namespace sa {

template <bool FAST>
__device__ __forceinline__ double sa_row(const dev::SellView& S, int t, const double* __restrict__ x) {
  double acc = 0.0;
  dev::for_each_entry(S, t, t, x, [&](int, double a, double xv) {
    acc = FAST ? __fma_rn(a, xv, acc) : __dadd_rn(acc, __dmul_rn(a, xv));
  });
  return acc;
}

template <bool FAST>
__global__ void __launch_bounds__(256) k_restrict_sa(dev::SellView R, const double* __restrict__ r,
                                                     double* __restrict__ f_coarse, double* __restrict__ u_coarse) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= R.n_rows) return;
  f_coarse[t] = sa_row<FAST>(R, t, r);
  if (u_coarse) u_coarse[t] = 0.0;
}

template <bool FAST>
__global__ void __launch_bounds__(256) k_prolong_add_sa(dev::SellView P, const double* __restrict__ e,
                                                        double* __restrict__ u) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= P.n_rows) return;
  const double pe = sa_row<FAST>(P, t, e);
  u[t] = __dadd_rn(u[t], pe);
}

}  // namespace sa
}  // namespace amgb
