// Device-side setup of a smoothed-aggregation hierarchy (AMGB_TRANSFER_SMOOTHED_AGGREGATION, sm_100a): the
// device counterparts of sa_aggregate's strength step, sa_prolongation, multiply (Galerkin products),
// transpose, bitwise_equal, build_dia and build_sell of host_setup.cpp.  Every value is formed with the
// host's operations in the host's order (explicit __d*_rn intrinsics, no contraction), so the levels
// and prolongators are bit-identical to the host build and to tests/oracle_sa.py.  The aggregation
// passes themselves stay sequential on the host (sa_aggregate_passes), on the downloaded strong graph.
// "Row i" of a matrix is its CSC column i throughout, as in host_setup.cpp.
#pragma once
#include <cstdint>

#include <cuda_runtime.h>

#include "setup_dia.cuh"

namespace amgb {
namespace sasetup {

// read-only CSC view of a device matrix
struct CscView {
  int rows, cols;
  const int* colptr;
  const int* rowidx;
  const double* val;
};

// ---- diagonal: d[i] = a_ii (0 when absent); *zero_row = lowest row with a zero diagonal (INT_MAX: none) ----
__global__ void __launch_bounds__(256) k_sa_diag(CscView A, double* __restrict__ d, int* zero_row) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= A.cols) return;
  double di = 0.0;
  for (int p = A.colptr[i]; p < A.colptr[i + 1]; ++p)
    if (A.rowidx[p] == i) di = A.val[p];
  d[i] = di;
  if (di == 0.0) atomicMin(zero_row, i);
}

// ---- strength graph: j != i is a strong neighbour of i when |a_ij| > theta sqrt(|a_ii| |a_jj|), a_ij != 0.
// FILL = false: cnt[i] = number of strong neighbours; FILL = true: snb[sptr[i]..] = them, ascending ----
template <bool FILL>
__global__ void __launch_bounds__(256) k_sa_strength(CscView A, const double* __restrict__ d, double theta,
                                                     long long* __restrict__ cnt, const long long* __restrict__ sptr,
                                                     int* __restrict__ snb) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= A.cols) return;
  const double di = fabs(d[i]);
  long long c = FILL ? sptr[i] : 0;
  for (int p = A.colptr[i]; p < A.colptr[i + 1]; ++p) {
    const int j = A.rowidx[p];
    const double a = A.val[p];
    if (j == i || a == 0.0) continue;
    const double thr = __dmul_rn(theta, __dsqrt_rn(__dmul_rn(di, fabs(d[j]))));
    if (fabs(a) > thr) {
      if (FILL) snb[c] = j;
      ++c;
    }
  }
  if (!FILL) cnt[i] = c;
}

// ---- Gershgorin bound of D^-1 A: max over rows of (sum of |a| over the stored entries, from +0 in
// ascending order) / |a_ii|.  The quotients are >= +0, so their bit patterns order like their values; a
// NaN quotient is skipped, as std::max(rho, NaN) keeps rho on the host ----
__global__ void __launch_bounds__(256) k_sa_gershgorin(CscView A, const double* __restrict__ d,
                                                       unsigned long long* rho_bits) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= A.cols) return;
  double s = 0.0;
  for (int p = A.colptr[i]; p < A.colptr[i + 1]; ++p) s = __dadd_rn(s, fabs(A.val[p]));
  const double r = __ddiv_rn(s, fabs(d[i]));
  if (r == r) atomicMax(rho_bits, (unsigned long long)__double_as_longlong(r));
}

// ---- smoothed prolongator, built as R = P^T (columns = fine rows i): on entry S(J, i) is the sum of the
// entries of row i whose column lies in aggregate J (from +0, ascending); on exit
// R(J, i) = T(i, J) - (w / a_ii) S(J, i) ----
__global__ void __launch_bounds__(256) k_sa_smooth(int n, const int* __restrict__ colptr, const int* __restrict__ rowidx,
                                                   double* __restrict__ val, const int* __restrict__ agg,
                                                   const double* __restrict__ d, double w) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double c = __ddiv_rn(w, d[i]);
  const int own = agg[i];
  for (int p = colptr[i]; p < colptr[i + 1]; ++p)
    val[p] = __dsub_rn(rowidx[p] == own ? 1.0 : 0.0, __dmul_rn(c, val[p]));
}

// ---- small helpers ----
__global__ void __launch_bounds__(256) k_iota(int* __restrict__ out, int64_t n) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) out[t] = (int)t;
}
__global__ void __launch_bounds__(256) k_fill(double* __restrict__ out, int64_t n, double v) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) out[t] = v;
}
template <class T>
__global__ void __launch_bounds__(256) k_narrow(const long long* __restrict__ in, T* __restrict__ out, int64_t n) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) out[t] = (T)in[t];
}
// col_of[p] = column of entry p
__global__ void __launch_bounds__(256) k_col_of(const int* __restrict__ colptr, int cols, int* __restrict__ col_of) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= cols) return;
  for (int p = colptr[c]; p < colptr[c + 1]; ++p) col_of[p] = c;
}
// entries per row (counts pre-zeroed)
__global__ void __launch_bounds__(256) k_row_count(const int* __restrict__ rowidx, int64_t nnz, long long* counts) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p < nnz) atomicAdd(reinterpret_cast<unsigned long long*>(counts + rowidx[p]), 1ull);
}
// transpose, after a stable sort of the entry numbers by row: entry q of the result is entry perm[q]
__global__ void __launch_bounds__(256) k_transpose_gather(const int* __restrict__ perm, const int* __restrict__ col_of,
                                                          const double* __restrict__ val, int64_t nnz,
                                                          int* __restrict__ t_rowidx, double* __restrict__ t_val) {
  const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= nnz) return;
  const int p = perm[q];
  t_rowidx[q] = col_of[p];
  t_val[q] = val[p];
}
// *differ = 1 when a and b differ in any bit
template <class T>
__global__ void __launch_bounds__(256) k_bits_differ(const T* __restrict__ a, const T* __restrict__ b, int64_t n,
                                                     int* differ) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  bool ne;
  if constexpr (sizeof(T) == 8)
    ne = __double_as_longlong(a[t]) != __double_as_longlong(b[t]);
  else
    ne = a[t] != b[t];
  if (ne) *differ = 1;
}

// ---- sparse product C = L R in Eigen's conservative order (host_setup.cpp: multiply) ----
// C(i, j) = sum over ascending k of L(i, k) R(k, j); the first term initialises the sum (PLUS_ZERO: the sum
// starts from +0 instead, as sa_prolongation's sums do), structural and computed zeros are kept.  One warp
// per output column j walks R's column j in order (ascending k) and its lanes share L's column k.  The rows
// of one L column are distinct, so within a step every accumulator is touched by one lane at most, and
// __syncwarp between steps makes each accumulator receive its terms in ascending k.  The accumulators are
// an open-addressing hash table of 2 x bound slots (at least 32), bound = min(L.rows, products of the
// column): in shared memory when it fits kSmallSlots, else in a per-warp global-memory table.  The
// symbolic pass counts the entries per column; the numeric pass writes them unsorted, and a segmented
// sort orders every column afterwards.
constexpr int kSmallSlots = 1024;  // shared slots per warp: bound <= kSmallSlots / 2
constexpr int kSpgemmWarps = 8;    // warps per block of the shared-memory pass
constexpr size_t kSpgemmSmem = (size_t)kSpgemmWarps * kSmallSlots * (sizeof(int) + sizeof(double));

// bound[j] = min(L.rows, sum over R(:, j) of the length of L(:, k)); the columns above `small_bound`
// are listed in big (in no particular order), the largest of their bounds goes to *max_big
__global__ void __launch_bounds__(256) k_spgemm_bound(CscView L, CscView R, long long* __restrict__ bound,
                                                      long long small_bound, int* __restrict__ big, int* n_big,
                                                      unsigned long long* max_big) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= R.cols) return;
  long long ub = 0;
  for (int q = R.colptr[j]; q < R.colptr[j + 1]; ++q) {
    const int k = R.rowidx[q];
    ub += L.colptr[k + 1] - L.colptr[k];
  }
  const long long b = ub < (long long)L.rows ? ub : (long long)L.rows;
  bound[j] = b;
  if (b > small_bound) {
    big[atomicAdd(n_big, 1)] = j;
    atomicMax(max_big, (unsigned long long)b);
  }
}

__device__ __forceinline__ int spgemm_slots(long long b) {
  int cap = 32;
  while ((long long)cap < 2 * b) cap <<= 1;
  return cap;
}

// list == nullptr: every column whose bound fits the shared table (the others are skipped); else the
// columns of list, with tables of g_slots slots per warp at g_keys / g_vals
template <bool NUMERIC, bool PLUS_ZERO>
__global__ void __launch_bounds__(kSpgemmWarps * 32, 2) k_spgemm(CscView L, CscView R, const long long* __restrict__ bound,
                                                              const int* __restrict__ list, int n_list, int* g_keys,
                                                              double* g_vals, int g_slots, long long* __restrict__ count,
                                                              const long long* __restrict__ cptr, int* __restrict__ c_rowidx,
                                                              double* __restrict__ c_val) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int64_t gw = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  int* keys;
  double* vals;
  if (list) {
    keys = g_keys + gw * (int64_t)g_slots;
    vals = g_vals + gw * (int64_t)g_slots;
  } else {
    vals = reinterpret_cast<double*>(smem) + w * kSmallSlots;
    keys = reinterpret_cast<int*>(smem + (size_t)kSpgemmWarps * kSmallSlots * sizeof(double)) + w * kSmallSlots;
  }
  const int64_t n_items = list ? n_list : R.cols;
  for (int64_t item = gw; item < n_items; item += n_warps) {
    const int j = list ? list[item] : (int)item;
    const long long b = bound[j];
    if (!list && 2 * b > kSmallSlots) continue;  // handled by the global-memory pass
    const int cap = spgemm_slots(b);
    const unsigned mask = (unsigned)cap - 1u;
    for (int s = lane; s < cap; s += 32) keys[s] = -1;
    __syncwarp();
    int inserted = 0;
    for (int q = R.colptr[j]; q < R.colptr[j + 1]; ++q) {
      const int k = R.rowidx[q];
      const double y = R.val[q];
      for (int p = L.colptr[k] + lane; p < L.colptr[k + 1]; p += 32) {
        const int i = L.rowidx[p];
        unsigned s = ((unsigned)i * 2654435761u) & mask;
        bool fresh = false;
        for (;;) {
          const int cur = *reinterpret_cast<volatile int*>(keys + s);
          if (cur == i) break;
          if (cur == -1) {
            const int old = atomicCAS(keys + s, -1, i);
            if (old == -1) {
              fresh = true;
              break;
            }
            if (old == i) break;
          }
          s = (s + 1) & mask;
        }
        if (NUMERIC) {
          const double term = __dmul_rn(L.val[p], y);
          vals[s] = fresh ? (PLUS_ZERO ? __dadd_rn(0.0, term) : term) : __dadd_rn(vals[s], term);
        } else {
          inserted += fresh;
        }
      }
      __syncwarp();
    }
    if (!NUMERIC) {
      inserted = __reduce_add_sync(0xffffffffu, inserted);
      if (lane == 0) count[j] = inserted;
    } else {
      long long out = cptr[j];
      for (int s0 = 0; s0 < cap; s0 += 32) {
        const int key = keys[s0 + lane];
        const unsigned has = __ballot_sync(0xffffffffu, key >= 0);
        if (key >= 0) {
          const long long at = out + __popc(has & ((1u << lane) - 1u));
          c_rowidx[at] = key;
          c_val[at] = vals[s0 + lane];
        }
        out += __popc(has);
      }
    }
    __syncwarp();
  }
}

// ---- CSC -> SELL-32 of "row c = CSC column c", explicit zeros dropped (host_setup.cpp: build_sell) ----
// len[c] = non-zero entries of column c; *nnz += their total
__global__ void __launch_bounds__(256) k_sell_len(CscView M, int* __restrict__ len, unsigned long long* nnz) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  int l = 0;
  if (c < M.cols)
    for (int p = M.colptr[c]; p < M.colptr[c + 1]; ++p) l += (M.val[p] != 0.0);
  if (c < M.cols) len[c] = l;
  const unsigned s = __reduce_add_sync(0xffffffffu, (unsigned)l);
  if ((threadIdx.x & 31) == 0 && s) atomicAdd(nnz, (unsigned long long)s);
}
// size[s] = 32 x the longest row of slice s
__global__ void __launch_bounds__(256) k_sell_slice_size(const int* __restrict__ len, int n, long long* __restrict__ size) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  const int l = t < n ? len[t] : 0;
  const int wmax = __reduce_max_sync(0xffffffffu, (unsigned)l);
  if ((threadIdx.x & 31) == 0 && t < n) size[t >> 5] = 32ll * wmax;
}
// col / val pre-filled with -1 / 0
__global__ void __launch_bounds__(256) k_sell_fill(CscView M, const long long* __restrict__ slice_off,
                                                   int* __restrict__ col, double* __restrict__ val) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= M.cols) return;
  const long long base = slice_off[t >> 5] + (t & 31);
  long long j = 0;
  for (int p = M.colptr[t]; p < M.colptr[t + 1]; ++p) {
    const double v = M.val[p];
    if (v == 0.0) continue;
    col[base + 32 * j] = M.rowidx[p];
    val[base + 32 * j] = v;
    ++j;
  }
}

// ---- CSC -> DIA over the non-zero entries only (build_dia ignores explicit zeros when it collects the
// offsets and leaves their slots +0): the counterparts of setup_dia.cuh's k_mark_offsets / k_csc_to_dia ----
__global__ void __launch_bounds__(256) k_mark_offsets_nz(CscView M, int shift, unsigned* bitmap) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= M.cols) return;
  for (int p = M.colptr[c]; p < M.colptr[c + 1]; ++p) {
    if (M.val[p] == 0.0) continue;
    const unsigned o = (unsigned)(M.rowidx[p] - c + shift);
    const unsigned bit = 1u << (o & 31u);
    if (!(bitmap[o >> 5] & bit)) atomicOr(bitmap + (o >> 5), bit);
  }
}
__global__ void __launch_bounds__(256) k_csc_to_dia_nz(const int* __restrict__ colptr, const int* __restrict__ rowidx,
                                                       const double* __restrict__ val, int n_cols, setup::Offsets off,
                                                       double* __restrict__ dia, int ld) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n_cols) return;
  for (int p = colptr[c]; p < colptr[c + 1]; ++p) {
    const double v = val[p];
    if (v == 0.0) continue;
    const int o = rowidx[p] - c;
#pragma unroll
    for (int d = 0; d < setup::kMaxOffsets; ++d)
      if (d < off.n && off.v[d] == o) dia[(size_t)d * ld + c] = v;
  }
}

}  // namespace sasetup
}  // namespace amgb
