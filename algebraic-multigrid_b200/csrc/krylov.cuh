// Krylov-basis kernels of amgb_solve_gmres (sm_100a): the classical Gram-Schmidt passes over a basis of
// k vectors stored in one allocation with leading dimension ld (a multiple of 32 doubles).
//
//   k_multidot    partial[i * nb + blk] = block blk's part of v_i . w, for i < k, in one pass: each block
//                 holds its tile of w in registers and streams the k basis tiles.
//   k_update<M>   out = base - sum_i c_i v_i (i ascending, base NULL means 0), with c in device memory;
//                 in the same pass M = kDots forms the partials of v_i . out (the reorthogonalisation),
//                 M = kSumSq those of out . out, M = kNone nothing.  t = V y is k_update<kNone> with no
//                 base and c = -y.
//   k_sum_rows    out[i] = sum of partial[i * nb + 0 .. nb), one block per i.
//
// Every sum runs in an order fixed by n alone (tile, warp, lane and block order), with no floating-point
// atomics, so two runs on the same data give identical bits.  FMAs are allowed: these kernels are not
// part of the oracle's bit-exact V-cycle.
#pragma once

#include <cstdint>

#include <cuda_runtime.h>

namespace amgb {
namespace krylov {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kPerThread = 4;                    // elements of w each thread holds
constexpr int kTile = kThreads * kPerThread;     // elements per block
constexpr int kGroup = 8;                        // dot products reduced together

enum Fused { kNone = 0, kDots = 1, kSumSq = 2 };

// blocks of k_multidot / k_update over n elements (the nb of the partial layout)
inline int tiles(int64_t n) { return n > 0 ? (int)((n + kTile - 1) / kTile) : 1; }
// leading dimension of the basis: n rounded up to 32 doubles (256 bytes)
inline int64_t basis_ld(int64_t n) { return (n + 31) / 32 * 32; }

// element e of thread t of block b: b * kTile + e * kThreads + t (coalesced per e)
__device__ __forceinline__ int64_t elem(int e) { return (int64_t)blockIdx.x * kTile + e * kThreads + threadIdx.x; }

// block sums of acc[0 .. cnt) (cnt <= kGroup) to partial[g * nb + blockIdx.x]
__device__ __forceinline__ void group_reduce(double (&acc)[kGroup], int cnt, double (*sh)[kWarps],
                                             double* __restrict__ partial, int nb) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int g = 0; g < kGroup; ++g) {
    double v = acc[g];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    if (lane == 0) sh[g][warp] = v;
  }
  __syncthreads();
  if (threadIdx.x < cnt) {
    double s = 0.0;
#pragma unroll
    for (int q = 0; q < kWarps; ++q) s += sh[threadIdx.x][q];
    partial[(int64_t)threadIdx.x * nb + blockIdx.x] = s;
  }
  __syncthreads();
}

// partials of v_i . w for i < k, w given by this thread's registers
__device__ __forceinline__ void tile_dots(const double* __restrict__ V, int64_t ld, int k,
                                          const double (&wr)[kPerThread], int64_t n, double (*sh)[kWarps],
                                          double* __restrict__ partial, int nb) {
  for (int i0 = 0; i0 < k; i0 += kGroup) {
    double acc[kGroup];
#pragma unroll
    for (int g = 0; g < kGroup; ++g) {
      acc[g] = 0.0;
      if (i0 + g < k) {
        const double* __restrict__ v = V + (int64_t)(i0 + g) * ld;
#pragma unroll
        for (int e = 0; e < kPerThread; ++e) {
          const int64_t x = elem(e);
          if (x < n) acc[g] = fma(__ldg(v + x), wr[e], acc[g]);
        }
      }
    }
    group_reduce(acc, min(kGroup, k - i0), sh, partial + (int64_t)i0 * nb, nb);
  }
}

__global__ void __launch_bounds__(kThreads) k_multidot(const double* __restrict__ V, int64_t ld, int k,
                                                       const double* __restrict__ w, int64_t n,
                                                       double* __restrict__ partial) {
  __shared__ double sh[kGroup][kWarps];
  double wr[kPerThread];
#pragma unroll
  for (int e = 0; e < kPerThread; ++e) {
    const int64_t x = elem(e);
    wr[e] = x < n ? w[x] : 0.0;
  }
  tile_dots(V, ld, k, wr, n, sh, partial, gridDim.x);
}

template <int M>
__global__ void __launch_bounds__(kThreads) k_update(double* out, const double* base,  // may be the same vector
                                                     const double* __restrict__ V, int64_t ld, int k,
                                                     const double* __restrict__ c, int64_t n,
                                                     double* __restrict__ partial) {
  __shared__ double sh[kGroup][kWarps];
  double wr[kPerThread];
#pragma unroll
  for (int e = 0; e < kPerThread; ++e) {
    const int64_t x = elem(e);
    wr[e] = (base && x < n) ? base[x] : 0.0;
  }
  int i = 0;
  for (; i + 4 <= k; i += 4) {  // four basis vectors in flight per thread
    const double c0 = -__ldg(c + i), c1 = -__ldg(c + i + 1), c2 = -__ldg(c + i + 2), c3 = -__ldg(c + i + 3);
    const double* __restrict__ v = V + (int64_t)i * ld;
#pragma unroll
    for (int e = 0; e < kPerThread; ++e) {
      const int64_t x = elem(e);
      if (x < n) {
        const double a0 = __ldg(v + x), a1 = __ldg(v + ld + x), a2 = __ldg(v + 2 * ld + x), a3 = __ldg(v + 3 * ld + x);
        wr[e] = fma(c3, a3, fma(c2, a2, fma(c1, a1, fma(c0, a0, wr[e]))));
      }
    }
  }
  for (; i < k; ++i) {
    const double ci = -__ldg(c + i);
    const double* __restrict__ v = V + (int64_t)i * ld;
#pragma unroll
    for (int e = 0; e < kPerThread; ++e) {
      const int64_t x = elem(e);
      if (x < n) wr[e] = fma(ci, __ldg(v + x), wr[e]);
    }
  }
#pragma unroll
  for (int e = 0; e < kPerThread; ++e) {
    const int64_t x = elem(e);
    if (x < n) out[x] = wr[e];
  }
  if (M == kDots) {
    tile_dots(V, ld, k, wr, n, sh, partial, gridDim.x);
  } else if (M == kSumSq) {
    double acc[kGroup] = {0.0};
#pragma unroll
    for (int e = 0; e < kPerThread; ++e) acc[0] = fma(wr[e], wr[e], acc[0]);
    group_reduce(acc, 1, sh, partial, gridDim.x);
  }
}

__global__ void __launch_bounds__(kThreads) k_sum_rows(const double* __restrict__ partial, int nb,
                                                       double* __restrict__ out) {
  __shared__ double sh[kWarps];
  const double* __restrict__ p = partial + (int64_t)blockIdx.x * nb;
  double s = 0.0;
  for (int q = threadIdx.x; q < nb; q += kThreads) s += p[q];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
#pragma unroll
    for (int q = 0; q < kWarps; ++q) t += sh[q];
    out[blockIdx.x] = t;
  }
}

// dst = src / d
__global__ void __launch_bounds__(kThreads) k_scale(double* __restrict__ dst, const double* __restrict__ src,
                                                    double d, int64_t n) {
  const int64_t x = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  if (x < n) dst[x] = src[x] / d;
}

// dst = -src (exact), so that a V-cycle on -v followed by 0 - A z gives A M(v)
__global__ void __launch_bounds__(kThreads) k_negate(double* __restrict__ dst, const double* __restrict__ src,
                                                     int64_t n) {
  const int64_t x = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  if (x < n) dst[x] = -src[x];
}

}  // namespace krylov
}  // namespace amgb
