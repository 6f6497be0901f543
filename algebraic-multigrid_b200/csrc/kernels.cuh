// Device kernels of the V-cycle path (sm_100a).  All of them are HBM-bound
// streaming kernels over a device mirror in one of two layouts (host_setup.hpp):
//   DIA      diagonal storage for banded operators (all levels of this path):
//            no index array, x gathers independent of any prior load;
//   SELL-32  sliced ELL with explicit column indices for everything else.
// One thread per matrix row, a warp per 32 consecutive rows, so every load of
// val (and col) is a full 256/128-byte coalesced request and, for banded
// operators, so are the gathers of x.  Each thread walks its row in ascending column
// order with explicit __dmul_rn/__dadd_rn/__dsub_rn/__ddiv_rn (never contracted
// into FMAs), which reproduces the reference's summation order bit for bit:
//   Gauss-Seidel update   include/amg/smoother.hpp:101-138
//   residual r = f - A u  include/amg/multigrid.hpp:272-274 (Eigen: r=f; r-=A*u)
//   restriction           include/amg/interpolator.hpp:64-68
//   prolongation + add    include/amg/interpolator.hpp:52-56, multigrid.hpp:294-296
//   rss                   include/amg/common.hpp:17-27
#pragma once
#include <cstdint>
#include <cuda_pipeline.h>
#include <cuda_runtime.h>

namespace amgb {
namespace dev {

struct SellView {
  int n_rows;                 // rows covered by this view
  int n_slices;
  const uint32_t* slice_ptr;  // n_slices + 1
  const int* col;             // -1 = padding
  const double* val;
  const int* rows;            // row ids when the view is a subset, else nullptr
};

constexpr int kMaxDiagDev = 16;
struct DiaView {
  int n_rows;   // rows covered by this view
  int c_min;    // x may be indexed in [c_min, c_max] relative to the pointer the kernel
  int c_max;    //   gets (full operator: [0, n-1]; row block: [-halo_lo, n_own+halo_hi-1])
  int ld;       // leading dimension of val (rows rounded up to 32)
  int n_diag;
  int off[kMaxDiagDev];  // ascending column offsets
  const double* val;     // val[d*ld + t], 0.0 = no entry
  const int* rows;       // row ids when the view is a subset, else nullptr
  // optional: bit d of mask[t >> 5] is clear when diagonal d has no entry in the 32-row
  // slice of row t, so the warp skips that 256-byte load (nullptr: all diagonals dense)
  const unsigned short* mask;
};

// Compile-time bound on the number of diagonals, so the walk below is fully
// unrolled and off[] is read straight from the constant bank.
template <int ND>
struct DiaViewT : DiaView {};

// Visit the entries of DIA row t (matrix row `row`) in ascending column order.
// All val loads and all x gathers are independent of each other (x index =
// row + off, clamped; an absent entry has val == 0 and is skipped).
template <int ND, class XLoad, class Fn>
__device__ __forceinline__ void for_each_entry_x(const DiaViewT<ND>& S, int t, int row, XLoad&& xload, Fn&& fn) {
  const double* vp = S.val + t;
  double v[ND], xv[ND];
  const unsigned m = S.mask ? S.mask[t >> 5] : 0xffffu;
#pragma unroll
  for (int d = 0; d < ND; ++d) v[d] = (d < S.n_diag && ((m >> d) & 1u)) ? vp[(size_t)d * S.ld] : 0.0;
#pragma unroll
  for (int d = 0; d < ND; ++d)
    xv[d] = (d < S.n_diag && ((m >> d) & 1u)) ? xload(min(max(row + S.off[d], S.c_min), S.c_max)) : 0.0;
#pragma unroll
  for (int d = 0; d < ND; ++d)
    if (v[d] != 0.0) fn(row + S.off[d], v[d], xv[d]);
}
template <int ND, class Fn>
__device__ __forceinline__ void for_each_entry(const DiaViewT<ND>& S, int t, int row, const double* x, Fn&& fn) {
  for_each_entry_x(S, t, row, [&](int c) { return x[c]; }, fn);
}

// Visit the entries of SELL row t in ascending column order.  Loads are
// batched four at a time (4 col + 4 val loads in flight, then 4 gathers).
template <class XLoad, class Fn>
__device__ __forceinline__ void for_each_entry_x(const SellView& S, int t, int /*row*/, XLoad&& xload, Fn&& fn) {
  const int s = t >> 5;
  const uint32_t begin = S.slice_ptr[s] + (t & 31);
  const uint32_t end = S.slice_ptr[s + 1];
  for (uint32_t p = begin; p < end; p += 128) {
    int c[4];
    double v[4], xv[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const uint32_t q = p + 32u * k;
      c[k] = (q < end) ? S.col[q] : -1;
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const uint32_t q = p + 32u * k;
      v[k] = (c[k] >= 0) ? S.val[q] : 0.0;
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) xv[k] = (c[k] >= 0) ? xload(c[k]) : 0.0;
#pragma unroll
    for (int k = 0; k < 4; ++k)
      if (c[k] >= 0) fn(c[k], v[k], xv[k]);
  }
}
template <class Fn>
__device__ __forceinline__ void for_each_entry(const SellView& S, int t, int row, const double* x, Fn&& fn) {
  for_each_entry_x(S, t, row, [&](int c) { return x[c]; }, fn);
}

// ((f - a1 x1) - a2 x2) - ...   (multigrid.hpp:272-274)
template <class M>
__device__ __forceinline__ double row_residual(const M& S, int t, int row, const double* x, double f) {
  double acc = f;
  for_each_entry(S, t, row, x, [&](int, double a, double xv) { acc = __dsub_rn(acc, __dmul_rn(a, xv)); });
  return acc;
}

// The reference's Gauss-Seidel row update (smoother.hpp:101-138): rsum from +0,
// off-diagonal terms added in ascending order, (b - rsum) / diag, skipped when
// the diagonal is zero or absent.
template <class M>
__device__ __forceinline__ double row_gs(const M& S, int t, int row, const double* x, double b,
                                         double keep) {
  double rsum = 0.0, diag = 0.0;
  for_each_entry(S, t, row, x, [&](int c, double a, double xv) {
    if (c == row) diag = a;
    else rsum = __dadd_rn(rsum, __dmul_rn(a, xv));
  });
  return (diag == 0.0) ? keep : __ddiv_rn(__dsub_rn(b, rsum), diag);
}

// i: global fine row; e[J - e_first] holds coarse entry J (e_first = global index of e[0],
// non-zero when the coarse vector is a halo-extended row block).
__device__ __forceinline__ double prolong_at(const double* __restrict__ e, int e_first, int n_coarse, int i) {
  double acc = 0.0;
  const int J = i >> 1;
  if (i & 1) {
    if (J >= 0 && J < n_coarse) acc = __dadd_rn(acc, __dmul_rn(1.0, e[J - e_first]));
  } else {
    if (J - 1 >= 0 && J - 1 < n_coarse) acc = __dadd_rn(acc, __dmul_rn(0.5, e[J - 1 - e_first]));
    if (J >= 0 && J < n_coarse) acc = __dadd_rn(acc, __dmul_rn(0.5, e[J - e_first]));
  }
  return acc;
}
// ------------------------------------------------------------------ damped Jacobi, fused variants
// First sweep from a zero initial guess (every coarse level starts its pre-smoothing from
// u = 0, multigrid.hpp:278): r = f - A*0 = f exactly, so u_new = 0 + omega*(f/d) = omega*(f/d)
// bit for bit, and neither the operator nor u is read.
template <int ND>
__global__ void __launch_bounds__(256) k_jacobi_zero(DiaViewT<ND> A, int diag_d, const double* __restrict__ f,
                                                     double omega, double* __restrict__ u_new) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= A.n_rows) return;
  const double diag = A.val[(size_t)diag_d * A.ld + t];
  u_new[t] = (diag == 0.0) ? 0.0 : __dmul_rn(omega, __ddiv_rn(f[t], diag));
}

// First post-smoothing sweep fused with the coarse-grid correction (multigrid.hpp:294-301):
// the sweep runs on u' = u + P e, with u'[c] = u[c] + (P e)[c] formed on the fly for every
// entry it reads, so u' is never written to memory.  fine_first = global row of u[0].
template <class M>
__global__ void __launch_bounds__(256) k_jacobi_prolong(M A, const double* __restrict__ u,
                                                        const double* __restrict__ e, int e_first, int n_coarse,
                                                        int fine_first, const double* __restrict__ f, double omega,
                                                        double* __restrict__ u_new) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= A.n_rows) return;
  auto corrected = [&](int c) { return __dadd_rn(u[c], prolong_at(e, e_first, n_coarse, fine_first + c)); };
  double acc = f[t], diag = 0.0;
  for_each_entry_x(A, t, t, corrected, [&](int c, double a, double xv) {
    if (c == t) diag = a;
    acc = __dsub_rn(acc, __dmul_rn(a, xv));
  });
  const double ut = corrected(t);
  u_new[t] = (diag == 0.0) ? ut : __dadd_rn(ut, __dmul_rn(omega, __ddiv_rn(acc, diag)));
}

// ------------------------------------------------------------------ residual
template <class M>
__global__ void __launch_bounds__(256) k_residual(M A, const double* __restrict__ u,
                                                  const double* __restrict__ f, double* __restrict__ r) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= A.n_rows) return;
  r[t] = row_residual(A, t, t, u, f[t]);
}

// ------------------------------------------------------------------ y = A x (generic operator)
// Eigen's ColMajor sparse x dense product as used by InterpolatorBase::restriction /
// prolongation (interpolator.hpp:52-68): y zero-initialised, every row accumulates its
// products in ascending column order from +0.  The view holds the ROWS of the operator.
template <class M>
__global__ void __launch_bounds__(256) k_spmv(M A, const double* __restrict__ x, double* __restrict__ y) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= A.n_rows) return;
  double acc = 0.0;
  for_each_entry(A, t, t, x, [&](int, double a, double xv) { acc = __dadd_rn(acc, __dmul_rn(a, xv)); });
  y[t] = acc;
}

// ------------------------------------------------------------------ damped Jacobi
// u_new[k] = u[k] + omega * (r_k / a_kk), r_k as in k_residual.
// Rows row0 .. (skipping [hole_begin, hole_begin + hole_len)) up to A.n_rows: the sharded
// V-cycle sweeps the interior of a row block while the halo exchange is in flight and the
// rows next to the block edges afterwards (one launch with a hole in the middle).
template <class M>
__global__ void __launch_bounds__(256) k_jacobi(M A, const double* __restrict__ u,
                                                const double* __restrict__ f, double omega,
                                                double* __restrict__ u_new, int row0, int hole_begin,
                                                int hole_len) {
  int t = row0 + blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= hole_begin) t += hole_len;
  if (t >= A.n_rows) return;
  double acc = f[t], diag = 0.0;
  for_each_entry(A, t, t, u, [&](int c, double a, double xv) {
    if (c == t) diag = a;
    acc = __dsub_rn(acc, __dmul_rn(a, xv));
  });
  const double ut = u[t];
  u_new[t] = (diag == 0.0) ? ut : __dadd_rn(ut, __dmul_rn(omega, __ddiv_rn(acc, diag)));
}

// ------------------------------------------------------------------ multicolour GS
// One colour: the view lists the rows of that colour; they only read other colours.
template <class M>
__global__ void __launch_bounds__(256) k_color_gs(M C, const double* __restrict__ f, double* u) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= C.n_rows) return;
  const int row = C.rows[t];
  u[row] = row_gs(C, t, row, u, f[row], u[row]);
}

// ------------------------------------------------------------------ level-scheduled GS
// Generic, bit-exact lexicographic Gauss-Seidel for any matrix: the rows of one
// wavefront of the (zero-pruned) dependency DAG are independent; fronts run in
// order inside ONE block (block barrier between fronts).  This is the fallback
// for operators the systolic kernel does not cover; it is latency-bound.
// entry walkers that read u with ld.global.cg (L2): values written by other
// threads of the block in an earlier front must be seen
template <class Fn>
__device__ __forceinline__ void for_each_entry_cg(const SellView& A, int row, const double* u, Fn&& fn) {
  const int s = row >> 5;
  const uint32_t begin = A.slice_ptr[s] + (row & 31), end = A.slice_ptr[s + 1];
  for (uint32_t p = begin; p < end; p += 32) {
    const int c = A.col[p];
    if (c < 0) break;
    fn(c, A.val[p], __ldcg(u + c));
  }
}
template <int ND, class Fn>
__device__ __forceinline__ void for_each_entry_cg(const DiaViewT<ND>& A, int row, const double* u, Fn&& fn) {
#pragma unroll
  for (int d = 0; d < ND; ++d) {
    if (d >= A.n_diag) break;
    const double a = A.val[(size_t)d * A.ld + row];
    if (a != 0.0) {
      const int c = row + A.off[d];
      fn(c, a, __ldcg(u + c));
    }
  }
}
template <class M>
__global__ void __launch_bounds__(1024) k_gs_fronts(M A, const int* __restrict__ order,
                                                    const int* __restrict__ front_ptr, int n_fronts,
                                                    const double* __restrict__ f, double* u) {
  for (int fr = 0; fr < n_fronts; ++fr) {
    const int b = front_ptr[fr], e = front_ptr[fr + 1];
    for (int i = b + threadIdx.x; i < e; i += blockDim.x) {
      const int row = order[i];
      double rsum = 0.0, diag = 0.0;
      for_each_entry_cg(A, row, u, [&](int c, double a, double xv) {
        if (c == row) diag = a;
        else rsum = __dadd_rn(rsum, __dmul_rn(a, xv));
      });
      if (diag != 0.0) __stcg(u + row, __ddiv_rn(__dsub_rn(f[row], rsum), diag));
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------ banded line-scan GS
// Fast lexicographic Gauss-Seidel for the banded operators of this path.  A sweep
// (D + L) u_new = f - U u_old is split into
//   k_gs_rhs    g = f - (not-yet-updated side) * u_old      fully parallel, HBM-bound
//   k_gs_lines  (D + L) u = g  solved in sweep order by ONE block: rows are taken in
//               consecutive blocks of B <= (smallest far distance) rows, so every far
//               already-updated neighbour of a block lies in earlier blocks and is read
//               from a shared-memory ring of the most recent values; the distance-1 chain
//               u_k = (c_k - l_k u_{k-1}) / d_k inside the block is a first-order linear
//               recurrence solved by a parallel scan of affine maps (warp shuffles, then
//               across warps).  Coefficients of the next block are prefetched while the
//               current block is scanned.
// The update order is the reference's (smoother.hpp:148-174); the scan re-associates the
// arithmetic of the distance-1 chain, so results agree with the oracle to rounding
// (measured <= 1e-14 relative), not bit for bit -- k_gs_fronts is the bit-exact kernel.
// `pos` is the position in sweep order: row = pos (forward) or n-1-pos (backward).
struct GsLineDesc {
  int n;            // rows
  int dir;          // +1 forward, -1 backward
  int B;            // rows per block step (even, <= smallest far distance, <= 1024)
  int ring_mask;    // ring size - 1 (power of two >= B + largest far distance + 1)
  int n_far;        // far already-updated diagonals (<= 4)
  int far_dist[4];  // their distances in sweep order (> 1), in summation order
  int short_carry;  // 1: max|q|^32 is below fp64 resolution, a warp only needs its predecessor
  int np;           // padded length of the position-ordered arrays (multiple of 2, >= n + 2)
  // static coefficients in SWEEP-POSITION order (pos = row forward, n-1-row backward), so
  // one block step reads a contiguous, 16-byte aligned range of each: TMA bulk copies
  const double* dinv;  // 1 / a_kk (0 where the diagonal is zero or absent)
  const double* q;     // -(a_{k,prev} / a_kk), the distance-1 chain coefficient
  const double* far;   // n_far arrays of np entries
};

// g[row] = f[row] - sum over the not-yet-updated side (upper for a forward sweep, lower
// for a backward sweep) of a * u_old, ascending column order.
template <int ND>
__global__ void __launch_bounds__(256) k_gs_rhs(DiaViewT<ND> A, int dir, const double* __restrict__ u,
                                                const double* __restrict__ f, double* __restrict__ g) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= A.n_rows) return;
  const double* vp = A.val + t;
  double v[ND], xv[ND];
#pragma unroll
  for (int d = 0; d < ND; ++d) {
    const bool take = (d < A.n_diag) && (dir > 0 ? A.off[d] > 0 : A.off[d] < 0);
    v[d] = take ? vp[(size_t)d * A.ld] : 0.0;
    xv[d] = take ? u[min(max(t + A.off[d], A.c_min), A.c_max)] : 0.0;
  }
  double acc = f[t];
#pragma unroll
  for (int d = 0; d < ND; ++d)
    if (v[d] != 0.0) acc = __dsub_rn(acc, __dmul_rn(v[d], xv[d]));
  g[dir > 0 ? t : A.n_rows - 1 - t] = acc;  // sweep-position order
}

struct Affine {  // x -> p + q x
  double q, p;
};
__device__ __forceinline__ Affine compose(Affine later, Affine earlier) {
  return Affine{later.q * earlier.q, later.p + later.q * earlier.p};
}
__device__ __forceinline__ Affine warp_scan_affine(Affine a, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const double qo = __shfl_up_sync(0xffffffffu, a.q, o);
    const double po = __shfl_up_sync(0xffffffffu, a.p, o);
    if (lane >= o) a = compose(a, Affine{qo, po});
  }
  return a;
}

// ---- TMA 1-D bulk copy + mbarrier (sm_90+/sm_100a) ----
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t}" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void tma_load_1d(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_u32(dst)),
      "l"(src), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}

// One block, rows taken in sweep order in block steps of B.  Per step: the step's slices of
// g / dinv / q / far coefficients arrive by TMA (issued STAGES-1 steps ahead by thread 0);
// every thread owns R consecutive rows of the block: it forms c = g - sum far * u_new (ring),
// p = c * dinv, composes its R affine maps u_k = p_k + q_k u_{k-1}, the block scans the
// per-thread maps, and each thread replays its rows from the value entering it and publishes
// them to the ring and to global memory.  (R = 4: one warp scan per 128 rows -- the kernel is
// instruction-issue bound on its single SM, and the scan is the largest share.)
template <int STAGES, int R>
__global__ void __launch_bounds__(1024) k_gs_lines(GsLineDesc D, const double* __restrict__ g, double* u) {
  extern __shared__ __align__(16) double smem[];
  double* ring = smem;                  // ring_mask + 1 doubles: most recent new values by position
  double* wq = smem + D.ring_mask + 1;  // 32 warp totals (q)
  double* wp = wq + 32;                 // 32 warp totals (p)
  uint64_t* bars = reinterpret_cast<uint64_t*>(wp + 32);  // STAGES mbarriers (8 slots reserved)
  double* stage = wp + 32 + 8;          // STAGES x (3 + n_far) x B
  // The last warp of the block is the PRODUCER: its lane 0 issues the TMA copies STAGES-1 steps
  // ahead and waits for the next step's stage, off the critical path of the compute warps.
  const int T = blockDim.x - 32, t = threadIdx.x, lane = t & 31, warp = t >> 5, n_warps = T >> 5;
  const bool producer = (t >= T);
  const int n = D.n, B = D.B, n_arr = 3 + D.n_far;
  const int n_steps = (n + B - 1) / B;

  if (t == T) {
    for (int i = 0; i < STAGES; ++i) mbar_init(&bars[i], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  // positions before the start of the sweep are read with a zero coefficient: keep them finite
  for (int i = t; i <= D.ring_mask; i += blockDim.x) ring[i] = 0.0;
  __syncthreads();

  auto issue = [&](int step) {  // producer lane 0 only
    if (step >= n_steps) return;
    const int b0 = step * B;
    const int cnt = min(B, n - b0);
    const uint32_t bytes = (uint32_t)((cnt + 1) & ~1) * 8u;  // arrays are padded, b0 is even
    const int sidx = step % STAGES;
    double* dst = stage + (size_t)sidx * n_arr * B;
    // the stage buffer was last READ before the block barrier that ended the previous step; a
    // write-after-read across proxies needs only that ordering
    mbar_expect_tx(&bars[sidx], bytes * (uint32_t)n_arr);
    tma_load_1d(dst, g + b0, bytes, &bars[sidx]);
    tma_load_1d(dst + B, D.dinv + b0, bytes, &bars[sidx]);
    tma_load_1d(dst + 2 * B, D.q + b0, bytes, &bars[sidx]);
    for (int k = 0; k < D.n_far; ++k)
      tma_load_1d(dst + (3 + k) * B, D.far + (size_t)k * D.np + b0, bytes, &bars[sidx]);
  };
  if (t == T) {
    for (int st = 0; st < STAGES - 1; ++st) issue(st);
    mbar_wait(&bars[0], 0u);
  }
  __syncthreads();  // stage 0 has landed

  const int stage_stride = n_arr * B;
  const int i0 = t * R;  // first row of this thread inside the block
  // u is walked forwards or backwards in memory; pos = b0 + i0 + r
  double* const u0 = (D.dir > 0) ? u + i0 : u + (n - 1 - i0);
  const int ustep = (D.dir > 0) ? 1 : -1;
  int sidx = 0, phase = 0;
  for (int step = 0; step < n_steps; ++step) {
    int nsidx = sidx + 1, nphase = phase;
    if (nsidx == STAGES) {
      nsidx = 0;
      nphase ^= 1;
    }
    if (producer) {
      if (t == T) {
        issue(step + STAGES - 1);  // its buffer was released by the barrier ending step-1
        if (step + 1 < n_steps) mbar_wait(&bars[nsidx], (uint32_t)nphase);  // next step's stage has landed
      }
      if (!D.short_carry && n_warps > 1) {  // stay in step with the compute warps' barriers
        __syncthreads();
        __syncthreads();
      } else if (n_warps > 1) {
        __syncthreads();
      }
      __syncthreads();
      sidx = nsidx;
      phase = nphase;
      continue;
    }
    const int b0 = step * B;
    const double* src = stage + sidx * stage_stride + i0;
    Affine rows[R];
    Affine mine{1.0, 0.0};
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const int pos = b0 + i0 + r;
      Affine m{1.0, 0.0};  // identity for padding rows
      if (i0 + r < B && pos < n) {
        double c = src[r];
        const double dinv = src[B + r];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          if (k < D.n_far) {
            // absent entries are stored as 0 and the ring only ever holds finite values
            c = __dsub_rn(c, __dmul_rn(src[(3 + k) * B + r], ring[(pos - D.far_dist[k]) & D.ring_mask]));
          }
        }
        m.p = c * dinv;
        m.q = src[2 * B + r];
        if (dinv == 0.0) {  // zero / absent diagonal: the reference leaves u unchanged (smoother.hpp:136)
          m.p = u0[(long long)ustep * (b0 + r)];
          m.q = 0.0;
        }
      }
      rows[r] = m;
      mine = compose(m, mine);
    }
    const double carry = (b0 > 0) ? ring[(b0 - 1) & D.ring_mask] : 0.0;
    const Affine incl = warp_scan_affine(mine, lane);
    // exclusive prefix inside the warp
    Affine excl{__shfl_up_sync(0xffffffffu, incl.q, 1), __shfl_up_sync(0xffffffffu, incl.p, 1)};
    if (lane == 0) excl = Affine{1.0, 0.0};
    double in;  // value entering this warp
    if (n_warps == 1) {
      in = carry;
      __syncwarp();
    } else if (D.short_carry) {
      // |q|^32 <= 2^-60: what enters a warp from further back than its predecessor is below
      // the last bit, so the value entering warp w is the predecessor's own last value
      if (lane == 31) wp[warp] = incl.p;
      __syncthreads();  // also: every ring read of this step happened before this point
      in = (warp == 0) ? carry : wp[warp - 1];
    } else {
      if (lane == 31) {
        wq[warp] = incl.q;
        wp[warp] = incl.p;
      }
      __syncthreads();
      if (warp == 0) {
        Affine w{lane < n_warps ? wq[lane] : 1.0, lane < n_warps ? wp[lane] : 0.0};
        w = warp_scan_affine(w, lane);
        wq[lane] = w.q;
        wp[lane] = w.p;
      }
      __syncthreads();
      in = (warp == 0) ? carry : wp[warp - 1] + wq[warp - 1] * carry;
    }
    double x = excl.p + excl.q * in;  // value entering this thread's first row
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const int pos = b0 + i0 + r;
      if (i0 + r < B && pos < n) {
        x = rows[r].p + rows[r].q * x;
        ring[pos & D.ring_mask] = x;
        u0[(long long)ustep * (b0 + r)] = x;
      }
    }
    sidx = nsidx;
    phase = nphase;
    __syncthreads();  // ring complete, this step's stage buffer free, next stage visible
  }
}

// ------------------------------------------------------------------ fused residual + restriction
// f_c[J] = ((0 + .5 r[2J]) + 1 r[2J+1]) + .5 r[2J+2]  with r = f - A u never
// written to HBM; also zeroes the coarse solution (multigrid.hpp:272-282).
// (The first fine row of the view must be an even global row.)
// A block computes 256 consecutive fine residuals starting at fine row 252*b and emits the
// 126 coarse rows 126*b .. 126*b+125, whose three fine rows all lie inside; consecutive
// blocks overlap by four fine rows (1.6 % redundant work) so no thread does a second row.
constexpr int kRRCoarsePerBlock = 126;
template <class M>
__global__ void __launch_bounds__(256) k_residual_restrict(M A, const double* __restrict__ u,
                                                           const double* __restrict__ f,
                                                           double* __restrict__ f_coarse,
                                                           double* __restrict__ u_coarse, int n_coarse) {
  __shared__ double r[256];
  const int base = blockIdx.x * (2 * kRRCoarsePerBlock);
  const int t = threadIdx.x;
  const int row = base + t;
  r[t] = (row < A.n_rows) ? row_residual(A, row, row, u, f[row]) : 0.0;
  __syncthreads();
  if (t < kRRCoarsePerBlock) {
    const int J = blockIdx.x * kRRCoarsePerBlock + t;
    if (J < n_coarse) {
      const double a = __dmul_rn(0.5, r[2 * t]);
      const double b = __dadd_rn(a, r[2 * t + 1]);
      f_coarse[J] = __dadd_rn(b, __dmul_rn(0.5, r[2 * t + 2]));
      if (u_coarse) u_coarse[J] = 0.0;
    }
  }
}

// stand-alone restriction (interpolator.hpp:64-68), for the per-operator API
__global__ void __launch_bounds__(256) k_restrict(const double* __restrict__ r, int n_fine,
                                                  double* __restrict__ f_coarse, int n_coarse) {
  const int J = blockIdx.x * blockDim.x + threadIdx.x;
  if (J >= n_coarse) return;
  double acc = 0.0;
  const int i = 2 * J;
  if (i < n_fine) acc = __dadd_rn(acc, __dmul_rn(0.5, r[i]));
  if (i + 1 < n_fine) acc = __dadd_rn(acc, __dmul_rn(1.0, r[i + 1]));
  if (i + 2 < n_fine) acc = __dadd_rn(acc, __dmul_rn(0.5, r[i + 2]));
  f_coarse[J] = acc;
}

// ------------------------------------------------------------------ prolongation + correction add
// u[i] = u[i] + (P e)[i]; (P e)[2J+1] = 0 + 1 e[J]; (P e)[2J] = (0 + .5 e[J-1]) + .5 e[J]
// with the terms whose coarse index is outside [0, n_coarse) absent
// (interpolator.hpp:52-56,118-125; multigrid.hpp:294-296).
// Two fine rows (an even row 2J and the odd row 2J+1) per thread: one 16-byte load / store of
// u and the coarse entries e[J-1], e[J].  Needs fine_first even and u 16-byte aligned.
__global__ void __launch_bounds__(256) k_prolong_add2(const double* __restrict__ e, int e_first, int n_coarse,
                                                      double* __restrict__ u, int fine_first, int n_own) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;  // pair index
  const int t = 2 * p;
  if (t >= n_own) return;
  if (t + 1 < n_own) {
    double2 v = *reinterpret_cast<double2*>(u + t);
    v.x = __dadd_rn(v.x, prolong_at(e, e_first, n_coarse, fine_first + t));
    v.y = __dadd_rn(v.y, prolong_at(e, e_first, n_coarse, fine_first + t + 1));
    *reinterpret_cast<double2*>(u + t) = v;
  } else {
    u[t] = __dadd_rn(u[t], prolong_at(e, e_first, n_coarse, fine_first + t));
  }
}
// u points at this rank's first owned fine row (global row fine_first), n_own rows.
__global__ void __launch_bounds__(256) k_prolong_add(const double* __restrict__ e, int e_first, int n_coarse,
                                                     double* __restrict__ u, int fine_first, int n_own) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_own) return;
  u[t] = __dadd_rn(u[t], prolong_at(e, e_first, n_coarse, fine_first + t));
}

// ------------------------------------------------------------------ bilinear transfer (2-D grids)
// AMGB_TRANSFER_BILINEAR_2D on an m_h x m_h grid (DOF k = y*m_h + x), m_H = m_h / 2: coarse point
// (Y, X) restricts from / prolongs to the fine points (2Y + a, 2X + b), a, b in {0, 1, 2}, inside the
// grid, with weight w(a) * w(b), w = (.5, 1, .5) (P = P1 (x) P1, R = P^T).  Sums run over ascending
// column index from +0, as Eigen's sparse x dense product (the oracle's spmv) does; every weight is a
// power of two, so the products are exact and the result is bit-identical in both arithmetic modes.
__device__ __forceinline__ double bl_w(int a) { return a == 1 ? 1.0 : 0.5; }

// stand-alone restriction f_c = R r, one thread per coarse point
__global__ void __launch_bounds__(256) k_restrict2d(const double* __restrict__ r, int m_h,
                                                    double* __restrict__ f_coarse, int m_H) {
  const int X = blockIdx.x * blockDim.x + threadIdx.x, Y = blockIdx.y;
  if (X >= m_H) return;
  double acc = 0.0;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    const int y = 2 * Y + a;
    if (y >= m_h) break;
#pragma unroll
    for (int b = 0; b < 3; ++b) {
      const int x = 2 * X + b;
      if (x >= m_h) break;
      acc = __dadd_rn(acc, __dmul_rn(bl_w(a) * bl_w(b), r[(size_t)y * m_h + x]));
    }
  }
  f_coarse[(size_t)Y * m_H + X] = acc;
}

// Fused residual + restriction: f_c = R (f - A u), u_c = 0 (multigrid.hpp:272-282).  A block owns a
// tile of kRR2Y x kRR2X coarse points; it forms the residuals of the (2 kRR2Y + 1) x (2 kRR2X + 1)
// fine points under the tile in shared memory (k_residual's per-row arithmetic) and restricts from
// there, so r never reaches HBM.  Neighbouring tiles share one fine line / column: 17 x 129 residuals
// for 16 x 128 distinct ones, 7 % formed twice.
// Window: the block produces the coarse lines [Y_begin, Y_end) (global line numbers); local line 0 of
// u, f and the operator rows is global fine line y_first, local line 0 of f_coarse / u_coarse global
// coarse line Y_first.  Residuals are formed on the fine lines [2 Y_begin, 2 Y_end] only (those the
// coarse lines restrict from), so a rank of a sharded level reads its own lines, the ghost lines above
// them and one line of u either side.  The whole level is y_first = Y_first = Y_begin = 0, Y_end = m_H
// (2 m_H + 1 >= m_h: every line, as before).
constexpr int kRR2X = 64, kRR2Y = 8;
template <class M>
__global__ void __launch_bounds__(256) k_residual_restrict2d(M A, const double* __restrict__ u,
                                                             const double* __restrict__ f, int m_h, int y_first,
                                                             double* __restrict__ f_coarse,
                                                             double* __restrict__ u_coarse, int m_H, int Y_first,
                                                             int Y_begin, int Y_end) {
  constexpr int FX = 2 * kRR2X + 1, FY = 2 * kRR2Y + 1;
  __shared__ double r[FY * FX];
  const int X0 = blockIdx.x * kRR2X, Y0 = Y_begin + blockIdx.y * kRR2Y;
  const int x0 = 2 * X0, y0 = 2 * Y0;
  const int y_end = min(m_h, 2 * Y_end + 1);
  for (int p = threadIdx.x; p < FY * FX; p += blockDim.x) {
    const int fy = p / FX, fx = p - fy * FX;
    const int y = y0 + fy, x = x0 + fx;
    double v = 0.0;
    if (y < y_end && x < m_h) {
      const int row = (y - y_first) * m_h + x;
      v = row_residual(A, row, row, u, f[row]);
    }
    r[p] = v;
  }
  __syncthreads();
  for (int p = threadIdx.x; p < kRR2Y * kRR2X; p += blockDim.x) {
    const int ty = p / kRR2X, tx = p - ty * kRR2X;
    const int Y = Y0 + ty, X = X0 + tx;
    if (Y >= Y_end || X >= m_H) continue;
    double acc = 0.0;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      if (2 * Y + a >= m_h) break;
#pragma unroll
      for (int b = 0; b < 3; ++b) {
        if (2 * X + b >= m_h) break;
        acc = __dadd_rn(acc, __dmul_rn(bl_w(a) * bl_w(b), r[(2 * ty + a) * FX + 2 * tx + b]));
      }
    }
    const size_t J = (size_t)(Y - Y_first) * m_H + X;
    f_coarse[J] = acc;
    if (u_coarse) u_coarse[J] = 0.0;
  }
}

// (P e) at fine point (y, x): fine coordinate y takes coarse Y = (y - 1) / 2 with weight 1 when odd, and
// Y = y / 2 - 1, y / 2 (those inside the coarse grid) with weight .5 each when even; the terms are summed
// in ascending coarse index (Y-major).  Fully unrolled and predicated, so all loads are independent.
// e points at global coarse line Y_first (lines below it may be read from a halo: signed offsets).
__device__ __forceinline__ double prolong2d_at(const double* __restrict__ e, int m_H, int Y_first, int y, int x) {
  const int ylo = (y & 1) ? (y >> 1) : max((y >> 1) - 1, 0), yhi = (y & 1) ? (y >> 1) : min(y >> 1, m_H - 1);
  const int xlo = (x & 1) ? (x >> 1) : max((x >> 1) - 1, 0), xhi = (x & 1) ? (x >> 1) : min(x >> 1, m_H - 1);
  const double w = ((y & 1) ? 1.0 : 0.5) * ((x & 1) ? 1.0 : 0.5);
  double v[4];
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 2; ++j)
      v[2 * i + j] = (ylo + i <= yhi && xlo + j <= xhi) ? e[(long long)(ylo + i - Y_first) * m_H + xlo + j] : 0.0;
  double acc = 0.0;
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 2; ++j)
      if (ylo + i <= yhi && xlo + j <= xhi) acc = __dadd_rn(acc, __dmul_rn(w, v[2 * i + j]));
  return acc;
}

// u += P e on the fine lines [y_begin, y_end) (y_begin even): a thread owns fine column x of the two
// fine lines y_begin + 2 blockIdx.y and the one after it (an even and an odd line, which share their
// coarse lines), with every load issued before the first add.  Local line 0 of u is global fine line
// y_first, of e global coarse line Y_first; the whole level is y_first = Y_first = y_begin = 0, y_end = m_h.
__global__ void __launch_bounds__(256) k_prolong_add2d(const double* __restrict__ e, int m_H, int Y_first,
                                                       double* __restrict__ u, int m_h, int y_first, int y_begin,
                                                       int y_end) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = y_begin + 2 * blockIdx.y;
  if (x >= m_h) return;
  const bool two = y + 1 < y_end;
  const size_t k = (size_t)(y - y_first) * m_h + x;
  const double u0 = u[k], u1 = two ? u[k + m_h] : 0.0;
  const double a0 = prolong2d_at(e, m_H, Y_first, y, x), a1 = two ? prolong2d_at(e, m_H, Y_first, y + 1, x) : 0.0;
  u[k] = __dadd_rn(u0, a0);
  if (two) u[k + m_h] = __dadd_rn(u1, a1);
}

// ------------------------------------------------------------------ peer-memory halo exchange
// One launch per exchange site (the stand-alone exchange of the per-operator sharded path and of
// the out-of-cycle sites; the fused legs push their boundary rows themselves, stream_leg.cuh).
// Block 0 serves the lower neighbour (rank g-1), block 1 the upper one, in two phases:
//   1. ARRIVE: bump the neighbour's "arrived" flag for this site and wait for its bump of ours.
//      A rank arrives only after every earlier kernel of its stream has finished, so from here
//      on nobody still reads the halo rows this exchange overwrites (no write-after-read hazard
//      whatever vector the previous site used, e.g. odd sweep counts);
//   2. DATA: copy this rank's boundary rows straight into the neighbour's halo region
//      (peer-mapped pointer, stores travel over NVLink), release them system-wide, bump the
//      neighbour's "data" flag and wait for ours.
// Epochs live in device memory so a replayed CUDA graph keeps counting.  A wait that exceeds
// timeout_cycles sets *timed_out; the host turns that into an error (results are invalid).
struct HaloSide {
  double* peer_dst;               // where my rows go in the neighbour's vector (nullptr: no neighbour)
  const double* src;              // my boundary rows
  int count;                      // doubles to send
  unsigned long long* peer_flag;  // neighbour's flag pair for (site, the side I am on from its view)
  unsigned long long* my_flag;    // my flag pair the neighbour bumps: [0] arrived, [1] data
};
__device__ __forceinline__ void flag_release(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long flag_acquire(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
// spin until *p >= want; false (and *timed_out = 1) after timeout_cycles
__device__ __forceinline__ bool flag_wait(const unsigned long long* p, unsigned long long want,
                                          long long timeout_cycles, int* timed_out) {
  const long long t0 = clock64();
  while (flag_acquire(p) < want) {
    if (clock64() - t0 > timeout_cycles) {  // a neighbour died or stalled: do not hang the GPU
      *timed_out = 1;
      return false;
    }
    __nanosleep(20);
  }
  return true;
}
__global__ void __launch_bounds__(1024) k_halo_exchange(HaloSide lo, HaloSide hi, unsigned long long* epoch,
                                                       int* timed_out, long long timeout_cycles) {
  const HaloSide S = blockIdx.x == 0 ? lo : hi;
  if (S.peer_dst == nullptr) return;
  __shared__ unsigned long long e_sh;
  if (threadIdx.x == 0) {
    const unsigned long long e = epoch[blockIdx.x] + 1;
    epoch[blockIdx.x] = e;
    e_sh = e;
    flag_release(S.peer_flag + 0, e);                       // I have arrived at this site
    flag_wait(S.my_flag + 0, e, timeout_cycles, timed_out);  // so has the neighbour
  }
  __syncthreads();
  for (int i = threadIdx.x; i < S.count; i += blockDim.x) S.peer_dst[i] = S.src[i];
  // bar.sync orders every thread's peer stores before thread 0's release store below
  // (release is cumulative over what happens-before it), so one system-scope release suffices
  __syncthreads();
  if (threadIdx.x == 0) {
    flag_release(S.peer_flag + 1, e_sh);
    flag_wait(S.my_flag + 1, e_sh, timeout_cycles, timed_out);
  }
  __syncthreads();
}

// ------------------------------------------------------------------ peer-memory all-gather
// The first level below the sharded ones is replicated: every rank needs all of its right-hand side,
// each rank having produced one block of it.  One launch: the blocks of group r (blockIdx.x / kSlices)
// serve peer r -- ARRIVE handshake (the peer has finished every earlier kernel, so nobody still reads
// the vector this launch overwrites), then each block stores its slice of this rank's rows straight
// into the peer's copy over NVLink, the last one releases the DATA flag, and everybody waits for the
// peer's own DATA flag before the launch ends.  Replaces G grouped NCCL broadcasts.
constexpr int kGatherSlices = 4;
constexpr int kGatherMaxPeers = 7;
struct GatherPeer {
  double* dst;                          // peer's copy of the vector (element 0)
  unsigned long long* peer_flags;       // peer's flag pair for ME as the source: [0] arrived, [1] data
  const unsigned long long* my_flags;   // my flag pair for this peer as the source
  unsigned long long* epoch;            // launches done with this peer
  unsigned int* done;                   // slice counter (self-resetting)
};
struct GatherParams {
  int n_peers;
  const double* src;  // my copy of the vector
  int begin, count;   // my rows [begin, begin + count)
  int* timed_out;
  long long timeout_cycles;
  GatherPeer peer[kGatherMaxPeers];
};
__global__ void __launch_bounds__(512) k_allgather_push(const __grid_constant__ GatherParams P) {
  const GatherPeer& R = P.peer[blockIdx.x / kGatherSlices];
  const int slice = blockIdx.x % kGatherSlices;
  __shared__ unsigned long long e_sh;
  if (threadIdx.x == 0) {
    const unsigned long long e = *reinterpret_cast<volatile unsigned long long*>(R.epoch) + 1ull;
    e_sh = e;
    if (slice == 0) flag_release(R.peer_flags + 0, e);          // I have arrived
    flag_wait(R.my_flags + 0, e, P.timeout_cycles, P.timed_out);  // so has the peer
  }
  __syncthreads();
  const int per = (P.count + kGatherSlices - 1) / kGatherSlices;
  const int lo = P.begin + slice * per, hi = min(P.begin + P.count, lo + per);
  for (int i = lo + threadIdx.x; i < hi; i += blockDim.x) R.dst[i] = P.src[i];
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned prev = atomicAdd(R.done, 1u);
    if (prev + 1u == (unsigned)kGatherSlices) {  // every slice is stored and fenced
      *R.done = 0u;
      __threadfence();
      *R.epoch = e_sh;
      flag_release(R.peer_flags + 1, e_sh);
    }
    flag_wait(R.my_flags + 1, e_sh, P.timeout_cycles, P.timed_out);  // the peer's rows have landed here
  }
  __syncthreads();
}

// ------------------------------------------------------------------ rss = sum (b - A u)^2
// bhat_i accumulates from +0 in ascending column order, d = b_i - bhat_i
// (common.hpp:21-25).  The outer sum is a fixed-shape tree (deterministic; it
// differs from the reference's sequential sum only by rounding).
__device__ __forceinline__ double block_sum_256(double v, double* sh) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
  __syncthreads();
  double tot = 0.0;
  if (threadIdx.x < 32) {
    tot = (threadIdx.x < (blockDim.x >> 5)) ? sh[threadIdx.x] : 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) tot += __shfl_down_sync(0xffffffffu, tot, o);
  }
  return tot;  // valid in thread 0
}
template <class M>
__global__ void __launch_bounds__(256) k_rss_partial(M A, const double* __restrict__ u,
                                                     const double* __restrict__ b,
                                                     double* __restrict__ partial) {
  __shared__ double sh[32];
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  double sq = 0.0;
  if (t < A.n_rows) {
    double bhat = 0.0;
    for_each_entry(A, t, t, u, [&](int, double a, double xv) { bhat = __dadd_rn(bhat, __dmul_rn(a, xv)); });
    const double d = __dsub_rn(b[t], bhat);
    sq = __dmul_rn(d, d);
  }
  const double tot = block_sum_256(sq, sh);
  if (threadIdx.x == 0) partial[blockIdx.x] = tot;
}
__global__ void __launch_bounds__(256) k_sum_partials(const double* __restrict__ partial, int n,
                                                      double* __restrict__ out) {
  __shared__ double sh[32];
  double acc = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) acc += partial[i];
  const double tot = block_sum_256(acc, sh);
  if (threadIdx.x == 0) *out = tot;
}
// sum of squares of a vector (for the relative-residual criterion)
__global__ void __launch_bounds__(256) k_sumsq_partial(const double* __restrict__ x, int n,
                                                       double* __restrict__ partial) {
  __shared__ double sh[32];
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  const double v = (t < n) ? x[t] : 0.0;
  const double tot = block_sum_256(v * v, sh);
  if (threadIdx.x == 0) partial[blockIdx.x] = tot;
}

// ------------------------------------------------------------------ vector kernels of the PCG wrapper
// (SURVEY.md section 8f rank 2: the V-cycle as the preconditioner of conjugate gradients)
__global__ void __launch_bounds__(256) k_dot_partial(const double* __restrict__ x, const double* __restrict__ y,
                                                     int n, double* __restrict__ partial) {
  __shared__ double sh[32];
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  const double v = (t < n) ? x[t] * y[t] : 0.0;
  const double tot = block_sum_256(v, sh);
  if (threadIdx.x == 0) partial[blockIdx.x] = tot;
}
// y += a x
__global__ void __launch_bounds__(256) k_axpy(double* __restrict__ y, double a, const double* __restrict__ x, int n) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) y[t] = y[t] + a * x[t];
}
// p = z + beta p
__global__ void __launch_bounds__(256) k_xpay(double* __restrict__ p, const double* __restrict__ z, double beta,
                                              int n) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) p[t] = z[t] + beta * p[t];
}

// ------------------------------------------------------------------ coarsest solve
// x = (L D L^T)^{-1} f with the banded factor of host_setup.hpp, right-looking
// substitutions (multigrid.hpp:287-288).  One block; the vector lives in shared
// memory when it fits, else in global memory.  The per-entry update order is
// fixed (ascending pivot in the forward pass, descending in the backward pass).
__global__ void __launch_bounds__(1024) k_banded_ldlt_solve(const double* __restrict__ L,
                                                            const double* __restrict__ d, int n, int bw,
                                                            const double* __restrict__ f,
                                                            double* __restrict__ x_out, double* work,
                                                            int x_in_smem, int L_in_smem) {
  extern __shared__ double sm[];
  double* x = x_in_smem ? sm : work;
  const int ld = bw > 0 ? bw : 1;
  const double* Lp = L;
  if (L_in_smem) {
    double* sL = sm + (x_in_smem ? n : 0);
    for (size_t i = threadIdx.x; i < (size_t)n * ld; i += blockDim.x) sL[i] = L[i];
    Lp = sL;
  }
  for (int i = threadIdx.x; i < n; i += blockDim.x) x[i] = f[i];
  __syncthreads();
  for (int i = 0; i < n; ++i) {
    const double xi = x[i];
    for (int t = 1 + threadIdx.x; t <= bw; t += blockDim.x) {
      const int r = i + t;
      if (r < n) x[r] = __dsub_rn(x[r], __dmul_rn(Lp[(size_t)r * ld + (i - (r - bw))], xi));
    }
    __syncthreads();
  }
  for (int i = threadIdx.x; i < n; i += blockDim.x) x[i] = __ddiv_rn(x[i], d[i]);
  __syncthreads();
  for (int i = n - 1; i >= 0; --i) {
    const double xi = x[i];
    for (int t = 1 + threadIdx.x; t <= bw; t += blockDim.x) {
      const int c = i - t;
      if (c >= 0) x[c] = __dsub_rn(x[c], __dmul_rn(Lp[(size_t)i * ld + (c - (i - bw))], xi));
    }
    __syncthreads();
  }
  for (int i = threadIdx.x; i < n; i += blockDim.x) x_out[i] = x[i];
}

// Same solve for half-bandwidth <= 31, run by ONE warp with the active part of the vector
// held in a register window (lane j holds the partial value of row pivot+j): per pivot one
// broadcast shuffle, one multiply-subtract and one shift shuffle, the factor entries and the
// entering element being read ahead of the dependent chain.  The order in which each entry
// receives its updates is that of k_banded_ldlt_solve, so the bits are the same.
__global__ void __launch_bounds__(32) k_banded_ldlt_solve_warp(const double* __restrict__ L,
                                                               const double* __restrict__ d, int n, int bw,
                                                               const double* __restrict__ f,
                                                               double* __restrict__ x_out, int L_in_smem) {
  extern __shared__ double sm[];
  double* y = sm;  // n
  const int lane = threadIdx.x;
  const int ld = bw > 0 ? bw : 1;
  const double* Lp = L;
  if (L_in_smem) {
    double* sL = sm + n;
    for (size_t i = lane; i < (size_t)n * ld; i += 32) sL[i] = L[i];
    Lp = sL;
  }
  __syncwarp();
  // the right-hand side is staged in shared memory once; factor entries and the element
  // entering the window are fetched one pivot ahead of the dependent shuffle chain
  for (int i = lane; i < n; i += 32) y[i] = f[i];
  __syncwarp();
  // forward: window lane j = partial x[i + j]
  double w = (lane < n) ? y[lane] : 0.0;
  auto fwd_l = [&](int i) {
    const int r = i + lane;
    return (lane >= 1 && lane <= bw && r < n) ? Lp[(size_t)r * ld + (bw - lane)] : 0.0;
  };
  double lij = fwd_l(0);
  double enter = (32 < n) ? y[32] : 0.0;
  for (int i = 0; i < n; ++i) {
    const double l_next = fwd_l(i + 1);
    const double e_next = (i + 33 < n) ? y[i + 33] : 0.0;
    const double xi = __shfl_sync(0xffffffffu, w, 0);
    if (lane == 0) y[i] = xi;  // rows <= i are final; the window has already consumed y[i]
    if (lij != 0.0) w = __dsub_rn(w, __dmul_rn(lij, xi));
    w = __shfl_down_sync(0xffffffffu, w, 1);
    if (lane == 31) w = enter;
    lij = l_next;
    enter = e_next;
  }
  __syncwarp();
  for (int i = lane; i < n; i += 32) y[i] = __ddiv_rn(y[i], d[i]);
  __syncwarp();
  // backward: window lane j = partial z[i - j]
  w = (n - 1 - lane >= 0) ? y[n - 1 - lane] : 0.0;
  auto bwd_l = [&](int i) {
    const int c = i - lane;
    return (i >= 0 && lane >= 1 && lane <= bw && c >= 0) ? Lp[(size_t)i * ld + (bw - lane)] : 0.0;
  };
  double lic = bwd_l(n - 1);
  enter = (n - 33 >= 0) ? y[n - 33] : 0.0;
  for (int i = n - 1; i >= 0; --i) {
    const double l_next = bwd_l(i - 1);
    const double e_next = (i - 33 >= 0) ? y[i - 33] : 0.0;
    const double xi = __shfl_sync(0xffffffffu, w, 0);
    if (lane == 0) x_out[i] = xi;
    if (lic != 0.0) w = __dsub_rn(w, __dmul_rn(lic, xi));
    w = __shfl_down_sync(0xffffffffu, w, 1);
    if (lane == 31) w = enter;
    lic = l_next;
    enter = e_next;
  }
}

// Same solve for half-bandwidth BW <= 8 as a plain recurrence: one thread keeps the last BW
// results in registers, so a row costs one short multiply-subtract chain instead of the
// shuffle round trips of the warp kernel.  Every entry receives its updates in the order of
// k_banded_ldlt_solve (ascending pivot forward, descending pivot backward), i.e. the oracle's
// order.  Factor and vector are staged in shared memory by all threads of the block (sm holds
// n * (BW + 1) doubles); the division pass is spread over the threads.  Block-wide call.
template <int BW>
__device__ __forceinline__ void ldlt_serial_block(double* sm, const double* __restrict__ L,
                                                  const double* __restrict__ d, int n,
                                                  const double* __restrict__ f, double* __restrict__ x_out) {
  double* y = sm;       // n
  double* sL = sm + n;  // n * BW
  const int t = threadIdx.x, T = blockDim.x;
  for (int i = t; i < n * BW; i += T) sL[i] = L[i];
  for (int i = t; i < n; i += T) y[i] = __ldcg(f + i);
  __syncthreads();
  if (t == 0) {
    double win[BW];  // win[k - 1] = y[r - k]
#pragma unroll
    for (int k = 0; k < BW; ++k) win[k] = 0.0;
#pragma unroll 4
    for (int r = 0; r < n; ++r) {
      double acc = y[r];
      const double* lr = sL + (size_t)r * BW;
#pragma unroll
      for (int k = BW; k >= 1; --k)
        if (r - k >= 0) acc = __dsub_rn(acc, __dmul_rn(lr[BW - k], win[k - 1]));
#pragma unroll
      for (int k = BW - 1; k >= 1; --k) win[k] = win[k - 1];
      win[0] = acc;
      y[r] = acc;
    }
  }
  __syncthreads();
  for (int i = t; i < n; i += T) y[i] = __ddiv_rn(y[i], d[i]);
  __syncthreads();
  if (t == 0) {
    double win[BW];  // win[k - 1] = x[c + k]
#pragma unroll
    for (int k = 0; k < BW; ++k) win[k] = 0.0;
#pragma unroll 4
    for (int c = n - 1; c >= 0; --c) {
      double acc = y[c];
#pragma unroll
      for (int k = BW; k >= 1; --k)
        if (c + k < n) acc = __dsub_rn(acc, __dmul_rn(sL[(size_t)(c + k) * BW + (BW - k)], win[k - 1]));
#pragma unroll
      for (int k = BW - 1; k >= 1; --k) win[k] = win[k - 1];
      win[0] = acc;
      y[c] = acc;
    }
  }
  __syncthreads();
  for (int i = t; i < n; i += T) x_out[i] = y[i];
  __syncthreads();
}
__device__ __forceinline__ void ldlt_serial_block_bw(int bw, double* sm, const double* L, const double* d, int n,
                                                     const double* f, double* x_out) {
  switch (bw) {
    case 1: ldlt_serial_block<1>(sm, L, d, n, f, x_out); break;
    case 2: ldlt_serial_block<2>(sm, L, d, n, f, x_out); break;
    case 3: ldlt_serial_block<3>(sm, L, d, n, f, x_out); break;
    case 4: ldlt_serial_block<4>(sm, L, d, n, f, x_out); break;
    case 5: ldlt_serial_block<5>(sm, L, d, n, f, x_out); break;
    case 6: ldlt_serial_block<6>(sm, L, d, n, f, x_out); break;
    case 7: ldlt_serial_block<7>(sm, L, d, n, f, x_out); break;
    default: ldlt_serial_block<8>(sm, L, d, n, f, x_out); break;
  }
}
__global__ void __launch_bounds__(128) k_banded_ldlt_solve_serial(const double* __restrict__ L,
                                                                  const double* __restrict__ d, int n, int bw,
                                                                  const double* __restrict__ f,
                                                                  double* __restrict__ x_out) {
  extern __shared__ double sm[];
  ldlt_serial_block_bw(bw, sm, L, d, n, f, x_out);
}

// ------------------------------------------------------------------ coarse tail of the V-cycle
// The levels below a size threshold hold a few thousand rows each: every kernel on them is pure
// launch latency (~4 us) and there are six per level.  This kernel runs the WHOLE tail of a
// damped-Jacobi cycle -- for every tail level the pre-smoothing sweeps, residual and
// restriction, then the coarsest solve, then for every tail level prolongation + add and the
// post-smoothing sweeps (multigrid.hpp:265-302) -- in ONE block, with block barriers where the
// per-operator kernels have launch boundaries.  Vectors stay in global memory (L2-resident);
// per-row arithmetic is that of k_jacobi_zero / k_jacobi / k_residual / k_restrict /
// k_prolong_add, so every bit is unchanged.
constexpr int kTailMaxLevels = 12;
struct TailLevel {
  DiaView A;   // rows of A (n_diag <= 10)
  int diag_d;  // index of the main diagonal
  int n, n_coarse;
  const double* f;
  double* u;
  double* tmp;
  double* f_coarse;  // next level's right-hand side
};
struct TailParams {
  int n_tail;   // tail levels that are smoothed (the coarsest level follows them)
  int nu;       // Jacobi sweeps per smooth call
  double omega;
  // coarsest level
  int nc, bw;
  const double* L;
  const double* d;
  const double* f_c;
  double* u_c;
  TailLevel lv[kTailMaxLevels];
};

// Vectors the block itself wrote earlier in the launch are read with ld.global.cg (L2), never
// through the non-coherent path.
template <int ND>
__device__ __forceinline__ void tail_jacobi(const TailLevel& V, const double* src, double* dst, double omega) {
  DiaViewT<ND> A;
  static_cast<DiaView&>(A) = V.A;
  for (int t = threadIdx.x; t < V.n; t += blockDim.x) {
    double acc = __ldcg(V.f + t), diag = 0.0;
    for_each_entry_x(A, t, t, [&](int c) { return __ldcg(src + c); }, [&](int c, double a, double xv) {
      if (c == t) diag = a;
      acc = __dsub_rn(acc, __dmul_rn(a, xv));
    });
    const double ut = __ldcg(src + t);
    dst[t] = (diag == 0.0) ? ut : __dadd_rn(ut, __dmul_rn(omega, __ddiv_rn(acc, diag)));
  }
}
template <int ND>
__device__ __forceinline__ void tail_residual(const TailLevel& V, const double* x, double* r) {
  DiaViewT<ND> A;
  static_cast<DiaView&>(A) = V.A;
  for (int t = threadIdx.x; t < V.n; t += blockDim.x) {
    double acc = __ldcg(V.f + t);
    for_each_entry_x(A, t, t, [&](int c) { return __ldcg(x + c); },
                     [&](int, double a, double xv) { acc = __dsub_rn(acc, __dmul_rn(a, xv)); });
    r[t] = acc;
  }
}

__global__ void __launch_bounds__(1024) k_coarse_tail(const __grid_constant__ TailParams P) {
  extern __shared__ double sm[];
  const int T = blockDim.x;
  // ---- down: u_l = 0 -> nu sweeps -> residual -> restriction.  Sweeps alternate tmp, u, tmp, ...
  // so that after the 2 nu sweeps of a whole cycle the iterate of the level sits in u.
  for (int l = 0; l < P.n_tail; ++l) {
    const TailLevel& V = P.lv[l];
    double* buf[2] = {V.tmp, V.u};
    for (int t = threadIdx.x; t < V.n; t += T) {  // first sweep from the zero guess (k_jacobi_zero)
      const double diag = V.A.val[(size_t)V.diag_d * V.A.ld + t];
      buf[0][t] = (diag == 0.0) ? 0.0 : __dmul_rn(P.omega, __ddiv_rn(__ldcg(V.f + t), diag));
    }
    __syncthreads();
    for (int s = 1; s < P.nu; ++s) {
      if (V.A.n_diag <= 6) tail_jacobi<6>(V, buf[(s - 1) & 1], buf[s & 1], P.omega);
      else tail_jacobi<10>(V, buf[(s - 1) & 1], buf[s & 1], P.omega);
      __syncthreads();
    }
    const double* x = buf[(P.nu - 1) & 1];
    double* r = buf[P.nu & 1];
    if (V.A.n_diag <= 6) tail_residual<6>(V, x, r);
    else tail_residual<10>(V, x, r);
    __syncthreads();
    for (int J = threadIdx.x; J < V.n_coarse; J += T) {  // k_restrict
      double acc = 0.0;
      const int i = 2 * J;
      if (i < V.n) acc = __dadd_rn(acc, __dmul_rn(0.5, __ldcg(r + i)));
      if (i + 1 < V.n) acc = __dadd_rn(acc, __dmul_rn(1.0, __ldcg(r + i + 1)));
      if (i + 2 < V.n) acc = __dadd_rn(acc, __dmul_rn(0.5, __ldcg(r + i + 2)));
      V.f_coarse[J] = acc;
    }
    __syncthreads();
  }
  // ---- coarsest solve (multigrid.hpp:287-288)
  ldlt_serial_block_bw(P.bw, sm, P.L, P.d, P.nc, P.f_c, P.u_c);
  // ---- up: x += P e, nu sweeps, result in u
  for (int l = P.n_tail - 1; l >= 0; --l) {
    const TailLevel& V = P.lv[l];
    double* buf[2] = {V.tmp, V.u};
    double* x = buf[(P.nu - 1) & 1];
    const double* e = (l + 1 < P.n_tail) ? P.lv[l + 1].u : P.u_c;
    for (int t = threadIdx.x; t < V.n; t += T) {
      double acc = 0.0;  // prolong_at with L2 loads
      const int J = t >> 1;
      if (t & 1) {
        if (J < V.n_coarse) acc = __dadd_rn(acc, __dmul_rn(1.0, __ldcg(e + J)));
      } else {
        if (J - 1 >= 0 && J - 1 < V.n_coarse) acc = __dadd_rn(acc, __dmul_rn(0.5, __ldcg(e + J - 1)));
        if (J < V.n_coarse) acc = __dadd_rn(acc, __dmul_rn(0.5, __ldcg(e + J)));
      }
      x[t] = __dadd_rn(__ldcg(x + t), acc);
    }
    __syncthreads();
    for (int s = 0; s < P.nu; ++s) {
      const double* src = buf[(P.nu - 1 + s) & 1];
      double* dst = buf[(P.nu + s) & 1];
      if (V.A.n_diag <= 6) tail_jacobi<6>(V, src, dst, P.omega);
      else tail_jacobi<10>(V, src, dst, P.omega);
      __syncthreads();
    }
  }
}

}  // namespace dev
}  // namespace amgb
