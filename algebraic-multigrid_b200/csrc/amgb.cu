// libamgb.so -- C ABI (include/amgb.h) over the sm_100a kernels of kernels.cuh.
// Holds the device mirrors (amgb_matrix, amgb_hierarchy), enqueues the V-cycle
// of include/amg/multigrid.hpp:263-305 on a stream and replays it as a CUDA
// graph.  There is no CPU fallback: every compute entry point needs a device.
#include "../../include/amgb.h"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_segmented_sort.cuh>
#include <cuda_runtime.h>

#include "host_setup.hpp"
#include "fused_leg.cuh"
#include "galerkin_dia.cuh"
#include "galerkin_dia2d.cuh"
#include "gs_wave.cuh"
#include "kernels.cuh"
#include "krylov.cuh"
#include "line_gs.cuh"
#include "mid_levels.cuh"
#include "setup_dia.cuh"
#include "setup_sa.cuh"
#include "transfer_sa.cuh"
#include "stream_leg_api.hpp"
#include "nccl_dyn.hpp"

namespace {

using namespace amgb;
using amgb::dev::DiaView;
using amgb::dev::SellView;

// A_H = R (A P) on the DIA layout, one thread per coarse row (galerkin_dia.cuh)
struct CoarseOffsets {
  int v[gal::kMaxDiag];
};
__global__ void __launch_bounds__(256) k_galerkin_dia(gal::FineDia A, int n_c, int nd_c, CoarseOffsets off_c,
                                                      double* __restrict__ val_c, int ld_c) {
  const int I = blockIdx.x * blockDim.x + threadIdx.x;
  if (I < n_c) gal::coarse_row(A, n_c, nd_c, off_c.v, I, val_c + I, ld_c);
}

// the same for the bilinear transfer of a 2-D hierarchy (galerkin_dia2d.cuh)
__global__ void __launch_bounds__(256) k_galerkin_dia2d(gal::FineDia A, int m_h, int m_H, int nd_c, CoarseOffsets off_c,
                                                        double* __restrict__ val_c, int ld_c) {
  const int I = blockIdx.x * blockDim.x + threadIdx.x;
  if (I < m_H * m_H) gal::coarse_row_2d(A, m_h, m_H, nd_c, off_c.v, I, val_c + I, ld_c);
}

thread_local std::string g_err;
std::atomic<int64_t> g_launches{0};

struct ApiError : std::runtime_error {
  int code;
  ApiError(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};

#define CUDA_CHECK(expr)                                                                   \
  do {                                                                                     \
    cudaError_t e_ = (expr);                                                               \
    if (e_ != cudaSuccess)                                                                 \
      throw ApiError(AMGB_ECUDA, std::string(#expr) + ": " + cudaGetErrorString(e_) + " (" + \
                                     __FILE__ + ":" + std::to_string(__LINE__) + ")");     \
  } while (0)

#define NCCL_CHECK(expr)                                                                  \
  do {                                                                                    \
    ncclResult_t r_ = (expr);                                                             \
    if (r_ != ncclSuccess)                                                                \
      throw ApiError(AMGB_ENCCL, std::string(#expr) + ": " + NcclApi::get().GetErrorString(r_) + \
                                     " (" + __FILE__ + ":" + std::to_string(__LINE__) + ")");   \
  } while (0)

#define LAUNCH(kernel, grid, block, smem, stream, ...)            \
  do {                                                            \
    kernel<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__);   \
    g_launches.fetch_add(1, std::memory_order_relaxed);           \
    CUDA_CHECK(cudaGetLastError());                               \
  } while (0)

template <class Fn>
int guarded(Fn&& fn) {
  try {
    fn();
    return AMGB_OK;
  } catch (const ApiError& e) {
    g_err = e.what();
    return e.code;
  } catch (const std::invalid_argument& e) {
    g_err = e.what();
    return AMGB_EINVAL;
  } catch (const std::exception& e) {
    g_err = e.what();
    return AMGB_ECUDA;
  }
}

void require_device() {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) {
    cudaGetLastError();
    throw ApiError(AMGB_ECUDA, "no CUDA device: libamgb has no CPU fallback");
  }
}

template <class T>
struct DevBuf {
  T* p = nullptr;
  size_t n = 0;
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  DevBuf(DevBuf&& o) noexcept : p(o.p), n(o.n) { o.p = nullptr; o.n = 0; }
  DevBuf& operator=(DevBuf&& o) noexcept {
    if (this != &o) { release(); p = o.p; n = o.n; o.p = nullptr; o.n = 0; }
    return *this;
  }
  ~DevBuf() { release(); }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    n = 0;
  }
  void alloc(size_t count) {
    release();
    n = count;
    CUDA_CHECK(cudaMalloc(&p, std::max<size_t>(count, 1) * sizeof(T)));
  }
  void zero(cudaStream_t s) { CUDA_CHECK(cudaMemsetAsync(p, 0, n * sizeof(T), s)); }
  void upload(const T* h, size_t count, cudaStream_t s) {
    if (count != n || !p) alloc(count);
    if (count) CUDA_CHECK(cudaMemcpyAsync(p, h, count * sizeof(T), cudaMemcpyHostToDevice, s));
  }
  void upload(const std::vector<T>& h, cudaStream_t s) { upload(h.data(), h.size(), s); }
  void download(T* h, cudaStream_t s) const {
    if (n) CUDA_CHECK(cudaMemcpyAsync(h, p, n * sizeof(T), cudaMemcpyDeviceToHost, s));
  }
};

struct DevSell {
  int n_rows = 0, n_slices = 0;
  int64_t nnz = 0;
  DevBuf<uint32_t> slice_ptr;
  DevBuf<int> col;
  DevBuf<double> val;
  DevBuf<int> rows;
  void upload(const Sell& S, cudaStream_t s) {
    n_rows = S.n_rows;
    n_slices = S.n_slices;
    nnz = S.nnz;
    slice_ptr.upload(S.slice_ptr, s);
    col.upload(S.col, s);
    val.upload(S.val, s);
    if (!S.rows.empty()) rows.upload(S.rows, s);
    CUDA_CHECK(cudaStreamSynchronize(s));  // host vectors may die after return
  }
  SellView view() const { return SellView{n_rows, n_slices, slice_ptr.p, col.p, val.p, rows.p}; }
};

struct DevDia {
  int n_rows = 0, c_min = 0, c_max = 0, ld = 0, n_diag = 0;
  int64_t nnz = 0;
  int off[dev::kMaxDiagDev] = {0};
  DevBuf<double> val;
  DevBuf<int> rows;
  DevBuf<unsigned short> mask;
  int64_t live_bytes = 0;  // matrix bytes a pass streams (masked-out slices excluded)
  void upload(const Dia& D, cudaStream_t s) {
    live_bytes = (int64_t)D.val.size() * 8;
    if (!D.mask.empty()) {
      mask.upload(D.mask, s);
      live_bytes = (int64_t)D.mask.size() * 2;
      for (unsigned short m : D.mask) live_bytes += 256ll * __builtin_popcount(m);
    }
    n_rows = D.n_rows;
    c_min = 0;
    c_max = D.n_cols - 1;
    ld = D.ld;
    n_diag = D.n_diag;
    nnz = D.nnz;
    for (int d = 0; d < n_diag; ++d) off[d] = D.off[d];
    val.upload(D.val, s);
    if (!D.rows.empty()) rows.upload(D.rows, s);
    CUDA_CHECK(cudaStreamSynchronize(s));
  }
  DiaView view() const {
    DiaView v;
    v.n_rows = n_rows;
    v.c_min = c_min;
    v.c_max = c_max;
    v.ld = ld;
    v.n_diag = n_diag;
    for (int d = 0; d < dev::kMaxDiagDev; ++d) v.off[d] = off[d];
    v.val = val.p;
    v.rows = rows.p;
    v.mask = mask.p;
    return v;
  }
};

// One device matrix: DIA when the operator is banded enough, else SELL-32.
struct DevMat {
  bool is_dia = false;
  DevDia dia;
  DevSell sell;
  void upload(const Csc& M, const std::vector<int>* rows, cudaStream_t s, bool allow_dia = true) {
    Dia D;
    if (allow_dia) D = build_dia(M, rows);
    is_dia = D.ok;
    if (is_dia) dia.upload(D, s);
    else sell.upload(build_sell(M, rows), s);
  }
  int n_rows() const { return is_dia ? dia.n_rows : sell.n_rows; }
  int64_t nnz() const { return is_dia ? dia.nnz : sell.nnz; }
  // bytes of matrix data one pass streams
  int64_t stored_bytes() const {
    return is_dia ? dia.live_bytes + (int64_t)dia.rows.n * 4
                  : (int64_t)sell.val.n * 12 + (int64_t)sell.slice_ptr.n * 4 + (int64_t)sell.rows.n * 4;
  }
};
// A CSC matrix on the device (explicit zeros kept): the levels and prolongators of the device-side
// smoothed-aggregation setup (setup_sa.cuh)
struct DevCsc {
  int rows = 0, cols = 0;
  int64_t nnz = 0;
  DevBuf<int> colptr, rowidx;
  DevBuf<double> val;
  sasetup::CscView view() const { return sasetup::CscView{rows, cols, colptr.p, rowidx.p, val.p}; }
  void upload(int r, int c, const int* cp, const int* ri, const double* v, cudaStream_t s) {
    rows = r;
    cols = c;
    nnz = cp[c];
    colptr.upload(cp, (size_t)c + 1, s);
    rowidx.upload(ri, (size_t)nnz, s);
    val.upload(v, (size_t)nnz, s);
    CUDA_CHECK(cudaStreamSynchronize(s));
  }
  Csc download(cudaStream_t s) const {
    Csc M;
    M.rows = rows;
    M.cols = cols;
    M.colptr.resize((size_t)cols + 1);
    M.rowidx.resize((size_t)nnz);
    M.val.resize((size_t)nnz);
    CUDA_CHECK(cudaMemcpyAsync(M.colptr.data(), colptr.p, M.colptr.size() * sizeof(int), cudaMemcpyDeviceToHost, s));
    if (nnz) {
      CUDA_CHECK(cudaMemcpyAsync(M.rowidx.data(), rowidx.p, nnz * sizeof(int), cudaMemcpyDeviceToHost, s));
      CUDA_CHECK(cudaMemcpyAsync(M.val.data(), val.p, nnz * sizeof(double), cudaMemcpyDeviceToHost, s));
    }
    CUDA_CHECK(cudaStreamSynchronize(s));
    return M;
  }
};

template <int ND>
dev::DiaViewT<ND> dia_view_t(const DevDia& d) {
  dev::DiaViewT<ND> v;
  static_cast<DiaView&>(v) = d.view();
  return v;
}
template <class Fn>
void with_view(const DevMat& m, Fn&& fn) {
  if (!m.is_dia) fn(m.sell.view());
  else if (m.dia.n_diag <= 6) fn(dia_view_t<6>(m.dia));
  else if (m.dia.n_diag <= 10) fn(dia_view_t<10>(m.dia));
  else fn(dia_view_t<16>(m.dia));
}

inline int blocks_for(int64_t n, int per_block) { return (int)((n + per_block - 1) / per_block); }

// Device mirror of one operator plus the lazily built smoother schedules.
struct Operator {
  Csc M;                  // structural CSC exactly as handed in (explicit zeros kept)
  Csc MT;                 // transpose (rows of A); built once
  bool symmetric = true;  // M == MT bitwise
  int n = 0;              // rows this rank smooths (all rows, or the owned block)
  int n_mat = 0;          // rows held on the device (n, or owned block + ghost rows)
  bool block = false;     // true: device holds a row block with local numbering
  DevMat colrows;                   // row c = CSC column c (smoother.hpp:101-117)
  std::unique_ptr<DevMat> arows;    // rows of A when !symmetric
  // generic Gauss-Seidel fronts
  bool have_fronts = false;
  DevBuf<int> f_order, f_ptr, b_order, b_ptr;
  int n_ffronts = 0, n_bfronts = 0;
  // banded line-scan Gauss-Seidel (k_gs_rhs + k_gs_lines)
  bool lines_checked = false, lines_ok = false;
  dev::GsLineDesc line_desc[2];  // [0] forward, [1] backward
  int lines_T = 0, lines_R = 0, lines_rows = 1;  // threads; TMA stages; rows per thread
  size_t lines_smem = 0;
  // multicolour
  bool have_colors = false;
  int n_colors = 0;
  std::vector<int> color;
  std::vector<std::unique_ptr<DevMat>> color_sell;

  void build(Csc&& A, cudaStream_t s) {
    if (A.rows != A.cols) throw std::invalid_argument("operator must be square");
    M = std::move(A);
    n = n_mat = M.cols;
    MT = transpose(M);
    symmetric = bitwise_equal(M, MT);
    colrows.upload(M, nullptr, s);
    if (!symmetric) {
      arows.reset(new DevMat());
      arows->upload(MT, nullptr, s);
    }
  }
  // Row-block mirror for a sharded level: rows [row_begin, row_begin + rows_stored) of A
  // in DIA with local numbering; x is indexed relative to the first owned row, the
  // halo-extended local vector allowing [-halo_lo, n_own + halo_hi - 1].
  void build_block(Csc&& A, int row_begin, int rows_stored, int n_own, int halo_lo, int halo_hi,
                   cudaStream_t s) {
    if (A.rows != A.cols) throw std::invalid_argument("operator must be square");
    M = std::move(A);
    MT = transpose(M);
    symmetric = bitwise_equal(M, MT);
    block = true;
    block_row0 = row_begin;
    n = n_own;
    n_mat = rows_stored;
    Dia D = build_dia_block(host_rows_of_A(), row_begin, rows_stored);
    if (!D.ok) throw std::invalid_argument("sharded levels need a banded operator (DIA layout)");
    colrows.is_dia = true;
    colrows.dia.upload(D, s);
    colrows.dia.c_min = -halo_lo;
    colrows.dia.c_max = n_own + halo_hi - 1;
  }
  // Window mirror for the fused legs of a sharded level: rows [row_begin, row_begin + n_rows) of A
  // (rows outside the level stay empty), diagonals ordered like the whole operator's.
  DevDia win;
  std::vector<int> win_off;
  bool build_window(int row_begin, int n_rows, cudaStream_t s) {
    const Csc& R = host_rows_of_A();
    std::vector<int> offs;
    for (int r = 0; r < R.cols; ++r)
      for (int p = R.colptr[r]; p < R.colptr[r + 1]; ++p) {
        if (R.val[p] == 0.0) continue;
        const int o = R.rowidx[p] - r;
        auto it = std::lower_bound(offs.begin(), offs.end(), o);
        if (it == offs.end() || *it != o) {
          if ((int)offs.size() == dev::kMaxDiagDev) return false;
          offs.insert(it, o);
        }
      }
    Dia D = build_dia_window(R, row_begin, n_rows, offs);
    if (!D.ok) return false;
    win.upload(D, s);
    win_off = offs;
    return true;
  }
  // Device-side setup: the level's rows-of-A DIA mirror was built on the GPU (setup_dia.cuh); no host
  // matrix is kept (M / MT stay empty, the hierarchy rebuilds them on demand for the getters).
  bool rows_primary = false;
  void adopt_rows(DevDia&& rowsA, int n_own_rows) {
    rows_primary = true;
    n = n_own_rows;
    n_mat = rowsA.n_rows;
    colrows.is_dia = true;
    colrows.dia = std::move(rowsA);
  }
  // the same with a rows-of-A mirror of either layout (device-side smoothed-aggregation setup)
  void adopt_rows(DevMat&& rowsA) {
    rows_primary = true;
    n = n_mat = rowsA.n_rows();
    colrows = std::move(rowsA);
  }
  const DevMat& rows_of_A() const { return (symmetric || block || rows_primary) ? colrows : *arows; }
  const Csc& host_rows_of_A() const { return symmetric ? M : MT; }  // CSC whose column k = row k of A

  void ensure_fronts(cudaStream_t s) {
    if (have_fronts) return;
    Schedule F = gs_schedule(M, true), B = gs_schedule(M, false);
    n_ffronts = F.n_fronts();
    n_bfronts = B.n_fronts();
    f_order.upload(F.order, s);
    f_ptr.upload(F.front_ptr, s);
    b_order.upload(B.order, s);
    b_ptr.upload(B.front_ptr, s);
    CUDA_CHECK(cudaStreamSynchronize(s));
    have_fronts = true;
  }
  // The line-scan kernel applies when the mirror is DIA and, on each side of the diagonal,
  // the entries are an optional distance-1 diagonal plus at most four "far" diagonals.
  // Builds, per direction, the sweep-position-ordered static arrays the kernel streams.
  DevBuf<double> line_coef[2];  // [dinv | q | far_0 .. far_{k-1}], each np entries
  void ensure_lines(cudaStream_t s) {
    if (lines_checked) return;
    lines_checked = true;
    if (!colrows.is_dia || block || n < 1) return;
    const DevDia& D = colrows.dia;
    bool has_diag = false;
    for (int d = 0; d < D.n_diag; ++d) has_diag |= (D.off[d] == 0);
    if (!has_diag) return;
    int B = 992, max_far = 0;  // 31 compute warps + the producer warp
    std::vector<int> dists[2];
    for (int side = 0; side < 2; ++side) {  // 0: forward (updated = lower), 1: backward (updated = upper)
      // ascending column order of the already-updated side: forward = most negative offset
      // first; backward = smallest positive offset first (the distance-1 entry goes to the scan)
      for (int d = 0; d < D.n_diag; ++d) {
        const int dist = side == 0 ? -D.off[d] : D.off[d];
        if (dist <= 1) continue;
        if (dists[side].size() == 4) return;
        dists[side].push_back(dist);
        B = std::min(B, dist);
        max_far = std::max(max_far, dist);
      }
    }
    B = std::min(B, n);
    B &= ~1;  // even: every step's slice starts on a 16-byte boundary (TMA)
    if (B < 2) return;
    lines_rows = 1;  // rows per thread (4 measured slower: bank conflicts, profiles/r1_gs_linescan.md)
    lines_T = ((B + lines_rows - 1) / lines_rows + 31) / 32 * 32;
    int ring = 64;
    while (ring < B + max_far + 1) ring <<= 1;
    const int n_far = (int)std::max(dists[0].size(), dists[1].size());
    const size_t cap = 220 * 1024;
    lines_R = 0;  // number of TMA stages
    for (int stages : {4, 3, 2}) {
      const size_t bytes = sizeof(double) * ((size_t)ring + 64 + 8 + (size_t)stages * (3 + n_far) * B);
      if (bytes <= cap) {
        lines_R = stages;
        lines_smem = bytes;
        break;
      }
    }
    if (lines_R == 0) return;
    const int np = ((n + 1) & ~1) + 2;
    for (int side = 0; side < 2; ++side) {
      const int nf = (int)dists[side].size();
      std::vector<double> coef((size_t)(2 + nf) * np, 0.0);
      double* dinv = coef.data();
      double* q = dinv + np;
      double qmax = 0.0;
      for (int k = 0; k < n; ++k) {
        const int pos = side == 0 ? k : n - 1 - k;
        double diag = 0.0, near = 0.0;
        for (int p = M.colptr[k]; p < M.colptr[k + 1]; ++p) {
          const double a = M.val[p];
          if (a == 0.0) continue;
          const int dist = side == 0 ? k - M.rowidx[p] : M.rowidx[p] - k;
          if (dist == 0) diag = a;
          else if (dist == 1) near = a;
          else if (dist > 1)
            for (int j = 0; j < nf; ++j)
              if (dists[side][j] == dist) coef[(size_t)(2 + j) * np + pos] = a;
        }
        dinv[pos] = diag != 0.0 ? 1.0 / diag : 0.0;
        q[pos] = diag != 0.0 ? -(near / diag) : 0.0;
        qmax = std::max(qmax, std::fabs(q[pos]));
      }
      line_coef[side].upload(coef, s);
      dev::GsLineDesc L{};
      L.n = n;
      L.dir = side == 0 ? +1 : -1;
      L.B = B;
      L.ring_mask = ring - 1;
      L.n_far = nf;
      for (int j = 0; j < nf; ++j) L.far_dist[j] = dists[side][j];
      L.short_carry = std::pow(qmax, 32.0) <= 0x1p-60 ? 1 : 0;  // below half an ulp of what it is added to
      L.np = np;
      L.dinv = line_coef[side].p;
      L.q = line_coef[side].p + np;
      L.far = line_coef[side].p + 2 * (size_t)np;
      line_desc[side] = L;
    }
    CUDA_CHECK(cudaStreamSynchronize(s));
    lines_ok = true;
  }
  // Multi-SM wavefront Gauss-Seidel (gs_wave.cuh), bit-identical to the reference's sweep: operators
  // whose entries couple neighbours of an n_lines x m grid and never cross the end of a line (level 0;
  // the Galerkin levels of the 1-D interpolation do cross it and stay with the line-scan kernel).
  bool wave_checked = false, wave_ok = false;
  gsw::Params wave_P[2];  // [0] forward, [1] backward
  int wave_S[2] = {0, 0};
  unsigned wave_mask = 0;  // stencil slots in use
  DevBuf<double> wave_coef[2], wave_hand;
  static bool wave_enabled() {
    static const bool on = [] {
      const char* e = std::getenv("AMGB_GS_WAVE");
      return !(e && std::atoi(e) == 0);
    }();
    return on;
  }
  void ensure_wave(cudaStream_t s) {
    if (wave_checked) return;
    wave_checked = true;
    if (!wave_enabled() || !colrows.is_dia || block || rows_primary || n < 9) return;
    const DevDia& D = colrows.dia;
    if (D.rows.p || D.n_rows != n || D.n_diag > gsw::kSlots) return;
    int cand[3];
    gsw::plan_candidates(D.off, D.n_diag, cand);
    DevBuf<unsigned> flags;  // [0] slots in use, [1] "an entry leaves the grid"
    flags.alloc(2);
    for (int ci = 0; ci < 3 && !wave_ok; ++ci) {
      const gsw::Plan Pl = gsw::plan_for(D.off, D.n_diag, n, cand[ci]);
      if (!Pl.ok) continue;
      gsw::CheckArgs C{};
      C.val = D.val.p;
      C.ld = D.ld;
      C.n_diag = D.n_diag;
      C.n = n;
      C.m = Pl.m;
      C.n_lines = Pl.n_lines;
      for (int d = 0; d < D.n_diag; ++d) C.e_of[d] = Pl.e_of[d];
      flags.zero(s);
      LAUNCH(gsw::k_gsw_check, blocks_for(n, 256), 256, 0, s, C, flags.p, reinterpret_cast<int*>(flags.p + 1));
      unsigned got[2] = {0, 0};
      CUDA_CHECK(cudaMemcpyAsync(got, flags.p, sizeof(got), cudaMemcpyDeviceToHost, s));
      CUDA_CHECK(cudaStreamSynchronize(s));
      if (got[1]) continue;
      const int n_blocks = (Pl.n_lines + gsw::kLinesPerBlock - 1) / gsw::kLinesPerBlock;
      gsw::Dia9 A9{};
      A9.val = D.val.p;
      A9.ld = D.ld;
      for (int e = 0; e < gsw::kSlots; ++e) A9.d_of[e] = Pl.d_of[e];
      bool fits = true;
      for (int side = 0; side < 2; ++side) {
        const int dir = side == 0 ? +1 : -1;
        const int S = gsw::stride_for(got[0], dir);
        const int T = Pl.m + S * 31;
        const int Ts = gsw::padded_steps(T);
        const size_t count = gsw::packed_doubles(n_blocks, T);
        if (count * sizeof(double) > (size_t)4 << 30) {  // packed copy of the operator: keep it sane
          fits = false;
          break;
        }
        wave_coef[side].alloc(count);
        wave_coef[side].zero(s);
        const long long threads = (long long)n_blocks * T * gsw::kLanes;
        LAUNCH(gsw::k_gsw_pack, (unsigned)((threads + 255) / 256), 256, 0, s, A9, n, Pl.m, Pl.n_lines, n_blocks, T, Ts,
               S, dir, wave_coef[side].p);
        gsw::Params P{};
        P.n = n;
        P.m = Pl.m;
        P.n_lines = Pl.n_lines;
        P.n_blocks = n_blocks;
        P.T = T;
        P.Ts = Ts;
        P.coef = wave_coef[side].p;
        P.timeout_cycles = 8000000000ll;  // ~4 s: a block whose predecessor died traps instead of hanging
        wave_P[side] = P;
        wave_S[side] = S;
      }
      if (!fits) {
        wave_coef[0].release();
        wave_coef[1].release();
        break;
      }
      wave_mask = got[0];
      wave_hand.alloc((size_t)n_blocks * Pl.m);
      for (int side = 0; side < 2; ++side) wave_P[side].hand = wave_hand.p;
      CUDA_CHECK(cudaStreamSynchronize(s));
      wave_ok = true;
    }
  }
  // AMGB_GS_WAVE_DIV=exact: __ddiv_rn inside the sweep; default: the split form of the same division
  // (gs_wave.cuh div_split), whose reciprocal part is evaluated when the operator is packed
  static bool wave_split_division() {
    const char* e = std::getenv("AMGB_GS_WAVE_DIV");
    return !(e && std::strcmp(e, "exact") == 0);
  }
  // look-ahead of the register ring in steps.  PD + 1 is a multiple of the three-deep neighbour
  // histories (the unrolled loop carries no moves); 5 steps cover an L2 miss of the per-lane f / u
  // lines, 2 steps (AMGB_GS_WAVE_PD=2) keep fewer loads in flight per scoreboard.
  static int wave_lookahead() {
    const char* e = std::getenv("AMGB_GS_WAVE_PD");
    return (e && std::atoi(e) == 2) ? 2 : 5;
  }
  template <bool SPLIT, int PD>
  static void (*pick_wave(bool five, int S, bool forward))(gsw::Params) {
    if (five) return forward ? gsw::k_gs_wave<1, 1, PD, gsw::kMaskFive, SPLIT> : gsw::k_gs_wave<1, -1, PD, gsw::kMaskFive, SPLIT>;
    if (S == 1) return forward ? gsw::k_gs_wave<1, 1, PD, gsw::kMaskAll, SPLIT> : gsw::k_gs_wave<1, -1, PD, gsw::kMaskAll, SPLIT>;
    return forward ? gsw::k_gs_wave<2, 1, PD, gsw::kMaskAll, SPLIT> : gsw::k_gs_wave<2, -1, PD, gsw::kMaskAll, SPLIT>;
  }
  void launch_wave(bool forward, const double* f, double* u, cudaStream_t s) {
    gsw::Params P = wave_P[forward ? 0 : 1];
    P.f = f;
    P.u = u;
    // the hand-over buffer starts as the sentinel (all bits set) on every sweep
    CUDA_CHECK(cudaMemsetAsync(wave_hand.p, 0xFF, wave_hand.n * sizeof(double), s));
    void (*kern)(gsw::Params) = nullptr;
    const int S = wave_S[forward ? 0 : 1];
    const bool five = (wave_mask & ~gsw::kMaskFive) == 0;  // five-point operator: half the stencil slots compile away
    const bool split = wave_split_division();
    if (wave_lookahead() == 2) kern = split ? pick_wave<true, 2>(five, S, forward) : pick_wave<false, 2>(five, S, forward);
    else kern = split ? pick_wave<true, 5>(five, S, forward) : pick_wave<false, 5>(five, S, forward);
    LAUNCH(kern, P.n_blocks, 32, 0, s, P);
  }
  // which kernel gs_direction runs for `mode`: 0 level-scheduled fronts, 1 line scan, 2 wavefront
  int gs_kernel(int mode, cudaStream_t s) {
    if (mode == AMGB_GS_AUTO) {
      ensure_wave(s);
      if (wave_ok) return AMGB_GS_KERNEL_WAVE;
    }
    if (mode == AMGB_GS_AUTO || mode == AMGB_GS_LINESCAN) {
      ensure_lines(s);
      if (lines_ok) return AMGB_GS_KERNEL_LINESCAN;
    }
    return AMGB_GS_KERNEL_FRONTS;
  }
  // one Gauss-Seidel direction (smoother.hpp:148-157 forward, :167-174 backward)
  void gs_direction(bool forward, const double* f, double* u, double* g_scratch, int mode, cudaStream_t s) {
    if (mode == AMGB_GS_AUTO) {
      ensure_wave(s);
      if (wave_ok) {
        launch_wave(forward, f, u, s);
        return;
      }
    }
    const bool scan = mode == AMGB_GS_AUTO || mode == AMGB_GS_LINESCAN;
    if (scan) ensure_lines(s);
    if (scan && lines_ok && g_scratch) {
      const dev::GsLineDesc& L = line_desc[forward ? 0 : 1];
      with_view(colrows, [&](auto V) { launch_gs_rhs(V, L.dir, u, f, g_scratch, s); });
      if (lines_rows == 4) {
        if (lines_R == 2) launch_gs_lines<2, 4>(L, g_scratch, u, s);
        else if (lines_R == 3) launch_gs_lines<3, 4>(L, g_scratch, u, s);
        else launch_gs_lines<4, 4>(L, g_scratch, u, s);
      } else {
        if (lines_R == 2) launch_gs_lines<2, 1>(L, g_scratch, u, s);
        else if (lines_R == 3) launch_gs_lines<3, 1>(L, g_scratch, u, s);
        else launch_gs_lines<4, 1>(L, g_scratch, u, s);
      }
    } else {
      ensure_fronts(s);
      if (forward) gs_forward(f, u, s);
      else gs_backward(f, u, s);
    }
  }
  template <int ND>
  void launch_gs_rhs(dev::DiaViewT<ND> V, int dir, const double* u, const double* f, double* g, cudaStream_t s) {
    auto kern = dev::k_gs_rhs<ND>;
    V.n_rows = n;
    LAUNCH(kern, blocks_for(n, 256), 256, 0, s, V, dir, u, f, g);
  }
  void launch_gs_rhs(SellView, int, const double*, const double*, double*, cudaStream_t) {
    throw ApiError(AMGB_ESTATE, "line-scan Gauss-Seidel needs the DIA layout");
  }
  template <int STAGES, int ROWS>
  void launch_gs_lines(const dev::GsLineDesc& L, const double* g, double* u, cudaStream_t s) {
    auto kern = dev::k_gs_lines<STAGES, ROWS>;
    static bool attr_done = false;
    if (!attr_done) {
      CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
      attr_done = true;
    }
    LAUNCH(kern, 1, lines_T + 32, lines_smem, s, L, g, u);  // + the producer warp
  }

  // Zebra line Gauss-Seidel (line_gs.cuh) on an m x m grid operator: per direction the factors
  // [sub | den (or 1 / den) | cp], each n doubles in step-major order, built on first use
  int lgs_m = 0;
  lgs::Grid lgs_grid{};
  DevBuf<double> lgs_fac[2];
  // `what` names the operator in the messages ("level 3"); throws std::invalid_argument when the
  // operator is not a 3 x 3 grid stencil or a line has a zero pivot
  void ensure_line_gs(int m, int D, bool fast, const std::string& what, cudaStream_t s) {
    if (lgs_fac[D].p) return;
    if (!lgs_m) {
      const DevMat& R = rows_of_A();
      if (m < 3)
        throw std::invalid_argument("line Gauss-Seidel needs at least 3 grid lines: " + what + " has " +
                                    std::to_string(m));
      const std::string no_grid = "line Gauss-Seidel: " + what + " is not an m x m grid operator with a 3 x 3 stencil "
                                  "that never couples across the end of a line";
      if (block || !R.is_dia || R.dia.rows.p || R.dia.n_rows != n || (int64_t)m * m != n)
        throw std::invalid_argument(no_grid);
      const DevDia& D9 = R.dia;
      const gsw::Plan Pl = gsw::plan_for(D9.off, D9.n_diag, n, m);
      if (!Pl.ok) throw std::invalid_argument(no_grid);
      gsw::CheckArgs C{};
      C.val = D9.val.p;
      C.ld = D9.ld;
      C.n_diag = D9.n_diag;
      C.n = n;
      C.m = m;
      C.n_lines = m;
      for (int d = 0; d < D9.n_diag; ++d) C.e_of[d] = Pl.e_of[d];
      DevBuf<unsigned> flags;  // [0] slots in use, [1] "an entry leaves the grid"
      flags.alloc(2);
      flags.zero(s);
      LAUNCH(gsw::k_gsw_check, blocks_for(n, 256), 256, 0, s, C, flags.p, reinterpret_cast<int*>(flags.p + 1));
      unsigned got[2] = {0, 0};
      CUDA_CHECK(cudaMemcpyAsync(got, flags.p, sizeof(got), cudaMemcpyDeviceToHost, s));
      CUDA_CHECK(cudaStreamSynchronize(s));
      if (got[1]) throw std::invalid_argument(no_grid);
      lgs_grid.val = D9.val.p;
      lgs_grid.ld = D9.ld;
      lgs_grid.m = m;
      for (int e = 0; e < gsw::kSlots; ++e) lgs_grid.d_of[e] = Pl.d_of[e];
      lgs_m = m;
    }
    DevBuf<double> fac;
    fac.alloc(3 * (size_t)n);
    DevBuf<int> bad;
    bad.alloc(1);
    const int none = INT_MAX;
    CUDA_CHECK(cudaMemcpyAsync(bad.p, &none, sizeof(int), cudaMemcpyHostToDevice, s));
    auto kern = fast ? lgs::k_line_factor<true> : lgs::k_line_factor<false>;
    LAUNCH(kern, blocks_for(m, 128), 128, 0, s, lgs_grid, D, fac.p, fac.p + n, fac.p + 2 * (size_t)n, bad.p);
    int row = none;
    CUDA_CHECK(cudaMemcpyAsync(&row, bad.p, sizeof(int), cudaMemcpyDeviceToHost, s));
    CUDA_CHECK(cudaStreamSynchronize(s));
    if (row != none)
      throw std::invalid_argument("line Gauss-Seidel: zero pivot in the " + std::string(D == lgs::kX ? "X" : "Y") +
                                  "-line solve of " + what + " at row " + std::to_string(row));
    lgs_fac[D] = std::move(fac);
  }
  // one pass: every line of direction D and colour c solved exactly (g: n scratch doubles)
  template <int D>
  void line_pass(int c, bool fast, const double* f, double* u, double* g, cudaStream_t s) const {
    const int m = lgs_m, nl = lgs::lines_of_colour(m, c);
    if (nl < 1) return;
    const double* fac = lgs_fac[D].p;
    if (fast) {
      LAUNCH((lgs::k_line_rhs<D, true>), blocks_for((int64_t)nl * m, 256), 256, 0, s, lgs_grid, c, f, u, g);
      LAUNCH((lgs::k_line_solve<D, true>), blocks_for(nl, lgs::kSolveThreads), lgs::kSolveThreads, 0, s, m, c, fac,
             fac + n, fac + 2 * (size_t)n, g, u);
    } else {
      LAUNCH((lgs::k_line_rhs<D, false>), blocks_for((int64_t)nl * m, 256), 256, 0, s, lgs_grid, c, f, u, g);
      LAUNCH((lgs::k_line_solve<D, false>), blocks_for(nl, lgs::kSolveThreads), lgs::kSolveThreads, 0, s, m, c, fac,
             fac + n, fac + 2 * (size_t)n, g, u);
    }
  }
  void line_pass(int D, int c, bool fast, const double* f, double* u, double* g, cudaStream_t s) const {
    if (D == lgs::kX) line_pass<lgs::kX>(c, fast, f, u, g, s);
    else line_pass<lgs::kY>(c, fast, f, u, g, s);
  }
  static int line_dirs(int lines, int* dirs) {
    if (lines == AMGB_LINES_Y) {
      dirs[0] = lgs::kY;
      return 1;
    }
    dirs[0] = lgs::kX;
    dirs[1] = lgs::kY;
    return lines == AMGB_LINES_ALTERNATING ? 2 : 1;
  }
  void ensure_line_gs_lines(int m, int lines, bool fast, const std::string& what, cudaStream_t s) {
    int dirs[2];
    const int nd = line_dirs(lines, dirs);
    for (int i = 0; i < nd; ++i) ensure_line_gs(m, dirs[i], fast, what, s);
  }
  // forward half: each direction in order, colour 0 then 1; backward half: reversed
  void line_gs_half(bool forward, int lines, bool fast, const double* f, double* u, double* g, cudaStream_t s) const {
    int dirs[2];
    const int nd = line_dirs(lines, dirs);
    for (int i = 0; i < nd; ++i) {
      const int D = dirs[forward ? i : nd - 1 - i];
      line_pass(D, forward ? 0 : 1, fast, f, u, g, s);
      line_pass(D, forward ? 1 : 0, fast, f, u, g, s);
    }
  }

  // first owned global row of a row block (0 for a whole level); the colour mirrors list GLOBAL rows
  int block_row0 = 0;
  void ensure_colors(cudaStream_t s) {
    if (have_colors) return;
    // the colouring is that of the WHOLE operator (every rank holds the host matrix), so a sharded
    // sweep visits the rows in the same colour order as one GPU does: same bits
    n_colors = greedy_coloring(M, MT, color);
    std::vector<std::vector<int>> members(n_colors);
    for (int k = block_row0; k < block_row0 + n; ++k) members[color[k]].push_back(k);
    color_sell.clear();
    for (int c = 0; c < n_colors; ++c) {
      color_sell.emplace_back(new DevMat());
      color_sell.back()->upload(host_rows_of_A(), &members[c], s);
    }
    have_colors = true;
  }

  // ---- launches (all asynchronous on s) ----
  void residual(const double* u, const double* f, double* r, cudaStream_t s) const {
    if (!n) return;
    with_view(rows_of_A(), [&](auto V) {
      auto kern = dev::k_residual<decltype(V)>;
      V.n_rows = n;
      LAUNCH(kern, blocks_for(n, 256), 256, 0, s, V, u, f, r);
    });
  }
  void jacobi(const double* u, const double* f, double omega, double* out, cudaStream_t s) const {
    if (!n) return;
    with_view(rows_of_A(), [&](auto V) {
      auto kern = dev::k_jacobi<decltype(V)>;
      V.n_rows = n;
      LAUNCH(kern, blocks_for(n, 256), 256, 0, s, V, u, f, omega, out, 0, n, 0);
    });
  }
  // rows [begin, end) only
  void jacobi_rows(const double* u, const double* f, double omega, double* out, int begin, int end,
                   cudaStream_t s) const {
    if (end <= begin) return;
    with_view(rows_of_A(), [&](auto V) {
      auto kern = dev::k_jacobi<decltype(V)>;
      V.n_rows = end;
      LAUNCH(kern, blocks_for(end - begin, 256), 256, 0, s, V, u, f, omega, out, begin, end, 0);
    });
  }
  // rows [0, lo) and [n - hi, n) in one launch
  void jacobi_edges(const double* u, const double* f, double omega, double* out, int lo, int hi,
                    cudaStream_t s) const {
    if (lo + hi <= 0) return;
    with_view(rows_of_A(), [&](auto V) {
      auto kern = dev::k_jacobi<decltype(V)>;
      V.n_rows = n;
      LAUNCH(kern, blocks_for(lo + hi, 256), 256, 0, s, V, u, f, omega, out, 0, lo, n - lo - hi);
    });
  }
  // first sweep from u = 0: only f and the diagonal are read (DIA); other layouts run the
  // ordinary sweep on an explicitly zeroed u
  bool jacobi_from_zero(const double* f, double omega, double* out, cudaStream_t s) const {
    const DevMat& A = rows_of_A();
    if (!n || !A.is_dia) return false;
    int diag_d = -1;
    for (int d = 0; d < A.dia.n_diag; ++d)
      if (A.dia.off[d] == 0) diag_d = d;
    if (diag_d < 0) return false;
    with_view(A, [&](auto V) { launch_jacobi_zero(V, diag_d, f, omega, out, s); });
    return true;
  }
  template <int ND>
  void launch_jacobi_zero(dev::DiaViewT<ND> V, int diag_d, const double* f, double omega, double* out,
                          cudaStream_t s) const {
    auto kern = dev::k_jacobi_zero<ND>;
    V.n_rows = n;
    LAUNCH(kern, blocks_for(n, 256), 256, 0, s, V, diag_d, f, omega, out);
  }
  void launch_jacobi_zero(SellView, int, const double*, double, double*, cudaStream_t) const {}
  // first post-smoothing sweep on u + P e without materialising it
  void jacobi_prolong(const double* u, const double* e, int e_first, int n_coarse, int fine_first,
                      const double* f, double omega, double* out, cudaStream_t s) const {
    if (!n) return;
    with_view(rows_of_A(), [&](auto V) {
      auto kern = dev::k_jacobi_prolong<decltype(V)>;
      V.n_rows = n;
      LAUNCH(kern, blocks_for(n, 256), 256, 0, s, V, u, e, e_first, n_coarse, fine_first, f, omega, out);
    });
  }
  void color_pass(int c, const double* f, double* u, cudaStream_t s) const {
    const DevMat& C = *color_sell[c];
    if (!C.n_rows()) return;
    with_view(C, [&](auto V) {
      auto kern = dev::k_color_gs<decltype(V)>;
      LAUNCH(kern, blocks_for(V.n_rows, 256), 256, 0, s, V, f, u);
    });
  }
  void gs_fronts(const int* order, const int* ptr, int n_fronts, const double* f, double* u,
                 cudaStream_t s) const {
    if (!n) return;
    with_view(colrows, [&](auto V) {
      auto kern = dev::k_gs_fronts<decltype(V)>;
      LAUNCH(kern, 1, 1024, 0, s, V, order, ptr, n_fronts, f, u);
    });
  }
  void gs_forward(const double* f, double* u, cudaStream_t s) const {
    gs_fronts(f_order.p, f_ptr.p, n_ffronts, f, u, s);
  }
  void gs_backward(const double* f, double* u, cudaStream_t s) const {
    gs_fronts(b_order.p, b_ptr.p, n_bfronts, f, u, s);
  }
  void residual_restrict(const double* u, const double* f, double* f_coarse, double* u_coarse,
                         int n_coarse, cudaStream_t s) const {
    with_view(rows_of_A(), [&](auto V) {
      auto kern = dev::k_residual_restrict<decltype(V)>;
      V.n_rows = n_mat;
      if (n_coarse > 0)
        LAUNCH(kern, blocks_for(n_coarse, dev::kRRCoarsePerBlock), 256, 0, s, V, u, f, f_coarse, u_coarse,
               n_coarse);
    });
  }
  // bilinear transfer of a 2-D hierarchy: this operator is the m_h x m_h grid level (or a block of it whose
  // first row is global line y_first), the coarse one m_H x m_H; produces coarse lines [Y_begin, Y_end) into
  // f_coarse / u_coarse, whose line 0 is global line Y_first
  void residual_restrict2d(const double* u, const double* f, int m_h, int y_first, double* f_coarse,
                           double* u_coarse, int m_H, int Y_first, int Y_begin, int Y_end, cudaStream_t s) const {
    if (m_H < 1 || Y_end <= Y_begin) return;
    with_view(rows_of_A(), [&](auto V) {
      auto kern = dev::k_residual_restrict2d<decltype(V)>;
      V.n_rows = n_mat;
      LAUNCH(kern, dim3(blocks_for(m_H, dev::kRR2X), blocks_for(Y_end - Y_begin, dev::kRR2Y)), 256, 0, s, V, u, f,
             m_h, y_first, f_coarse, u_coarse, m_H, Y_first, Y_begin, Y_end);
    });
  }
  int rss_blocks() const { return std::max(1, blocks_for(n, 256)); }
  // partial must hold rss_blocks() doubles; out one double
  void rss(const double* u, const double* b, double* partial, double* out, cudaStream_t s) const {
    const int nb = rss_blocks();
    with_view(rows_of_A(), [&](auto V) {
      auto kern = dev::k_rss_partial<decltype(V)>;
      V.n_rows = n;
      LAUNCH(kern, nb, 256, 0, s, V, u, b, partial);
    });
    LAUNCH(dev::k_sum_partials, 1, 256, 0, s, partial, nb, out);
  }
  int64_t nnz_device() const { return rows_of_A().nnz(); }
};

void options_default(amgb_options* o) {
  o->n_levels = 2;
  o->tolerance = 1e-9;
  o->compute_error_every_n_iters = 10;
  o->n_iters = 100;
  o->smoother = AMGB_SMOOTHER_GS;
  o->smoother_iters = 1;
  o->omega = 2.0 / 3.0;
  o->gs_mode = AMGB_GS_AUTO;
  o->use_graph = 1;
  o->skip_dead_coarse_smooth = 1;
  // zero-guess sweep, streaming legs, coarse tail, mid levels; prolongation fusion (bit 1) measured
  // slower.  The compressed operator formats (bit 6 matrix-free five-point legs, bit 7 row-type
  // dictionary legs) are opt-in: they apply to operators with verified structure only and turn the
  // legs from HBM-bound into issue-bound kernels (faster, but no longer a bandwidth roofline story);
  // AMGB_COMPRESS=1 switches them on for hierarchies created with the default options.
  o->fuse = 1 | 4 | 16 | 32;
  if (const char* c = std::getenv("AMGB_COMPRESS"))
    if (std::string(c) == "1") o->fuse |= 64 | 128;
  o->arith = AMGB_ARITH_REFERENCE;
  o->transfer = AMGB_TRANSFER_LINEAR;
  o->lines = AMGB_LINES_X;
  o->strength = 0.08;
  // the C++ mirror of the reference's headers has no argument for it: AMGB_ARITH=fast selects the fast
  // arithmetic for hierarchies created with the default options
  if (const char* a = std::getenv("AMGB_ARITH"))
    if (std::string(a) == "fast") o->arith = AMGB_ARITH_FAST;
}

}  // namespace

// ============================================================================
// amgb_matrix
// ============================================================================
struct amgb_matrix {
  int device = 0;
  cudaStream_t stream = nullptr;
  Operator op;
  DevBuf<double> u, b, r, partial, scalar;
  ~amgb_matrix() {
    if (stream) cudaStreamDestroy(stream);
  }
};

// ============================================================================
// amgb_comm: one NCCL communicator over the GPUs of one node (one rank per process)
// ============================================================================
struct amgb_comm {
  ncclComm_t comm = nullptr;
  int rank = 0, world = 1, device = 0;
  ~amgb_comm() {
    if (comm) NcclApi::get().CommDestroy(comm);
  }
};

// ============================================================================
// amgb_hierarchy
// ============================================================================
// Per-level state.  A level is either whole on this GPU (single-GPU run, or an
// agglomerated coarse level every rank keeps a replica of) or a contiguous row
// block [s, e) of a sharded fine level, with halo_lo / halo_hi extra entries of u
// below / above the block and `ghost` extra operator/rhs rows above it.
struct LevelState {
  bool sharded = false;
  int64_t n_global = 0;
  int64_t s = 0, e = 0;
  int halo_lo = 0, halo_hi = 0;
  int n_own = 0;  // e - s
  int n_mat = 0;  // operator / rhs rows held: n_own (+ ghost rows, clipped at the last row)
  DevBuf<double> u, f, tmp;
  DevBuf<double> fw;  // sharded levels with fused legs: f on the whole window [s - halo_lo, e + halo_hi)
  double* u_own() const { return u.p + halo_lo; }
  double* tmp_own() const { return tmp.p + halo_lo; }
  int64_t n_vec() const { return (int64_t)halo_lo + n_own + halo_hi; }
};

struct amgb_hierarchy {
  int device = 0;
  amgb_options opt{};
  int L = 0;
  std::vector<int64_t> n;
  std::vector<int64_t> m;  // grid lines per level of a 2-D hierarchy (n[l] = m[l]^2), empty otherwise
  bool bilinear() const { return opt.transfer == AMGB_TRANSFER_BILINEAR_2D; }
  bool sa() const { return opt.transfer == AMGB_TRANSFER_SMOOTHED_AGGREGATION; }
  // smoothed aggregation: P_l on the host, and on the device the rows of R_l = P_l^T (the CSC columns
  // of P_l) and the rows of P_l, both SELL-32
  std::vector<Csc> sa_P;
  std::vector<DevSell> sa_R_rows, sa_P_rows;
  // device-side setup with the damped-Jacobi smoother: the level operators and P_l stay on the device as
  // structural CSC (explicit zeros kept); the getters download them on demand into host_mats / a copy
  bool sa_resident = false;
  std::vector<DevCsc> sa_dev_A, sa_dev_P;
  // seconds of [strength + aggregation, prolongators, Galerkin products, mirrors + coarsest factor]
  double sa_times[4] = {0.0, 0.0, 0.0, 0.0};
  std::vector<std::unique_ptr<Operator>> ops;
  std::vector<LevelState> lv;
  DevBuf<double> partial, scalar;
  BandedLdlt factor;
  DevBuf<double> dL, dd, dwork;
  cudaStream_t own_stream = nullptr;
  cudaStream_t stream = nullptr;
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t exec = nullptr;
  int64_t launches_per_vcycle = 0;
  bool ldlt_attr_set = false, ldlt_warp_attr_set = false;
  int64_t iters_done = 0;
  std::vector<double> history;
  // sharding
  amgb_comm* comm = nullptr;  // borrowed
  PartitionPlan plan;
  int n_sharded = 0;
  int64_t halo_exchanges_per_vcycle = 0;
  // peer-memory halo exchange (CUDA IPC): per sharded level and vector (0 = u, 1 = tmp) the
  // neighbours' base pointers, plus epoch flags; falls back to NCCL send/recv when unavailable
  bool p2p = false;
  struct PeerMap {
    double* lo[3] = {nullptr, nullptr, nullptr};  // rank g-1's u / tmp / fw base
    double* hi[3] = {nullptr, nullptr, nullptr};  // rank g+1's u / tmp / fw base
    int lo_halo_lo = 0, lo_n_own = 0;    // geometry of rank g-1's block on this level
  };
  std::vector<PeerMap> peers;
  std::vector<void*> ipc_opened;
  DevBuf<unsigned long long> flags;      // [site][2]: bumped by the lower / upper neighbour
  unsigned long long* peer_flags_lo = nullptr;  // rank g-1's flags array
  unsigned long long* peer_flags_hi = nullptr;  // rank g+1's flags array
  DevBuf<unsigned long long> epochs;     // [site][2]
  // set by a kernel whose wait for a neighbour gave up; pinned host memory mapped into the device,
  // so the host checks it after every synchronise without a copy
  int* timed_out_host = nullptr;
  int* timed_out_dev = nullptr;
  long long halo_timeout_cycles = 8000000000ll;  // ~4 s of clock64; AMGB_HALO_TIMEOUT_MS overrides
  int n_sites = 0, site_cursor = 0;
  static constexpr int kMaxSites = 4096;
  static constexpr int kMaxLegSites = 64;  // fused legs: one site per sharded level and leg
  DevBuf<unsigned long long> leg_epochs;   // [leg site][side]
  DevBuf<unsigned int> leg_done;           // [leg site][side]
  bool fused_push = false;                 // the legs push their boundary rows themselves (no exchange launches)
  // peer-memory all-gather of the first replicated right-hand side (k_allgather_push)
  DevBuf<unsigned long long> gather_epochs;
  DevBuf<unsigned int> gather_done;
  dev::GatherParams gatherp{};
  bool gather_push = false;
  // second stream: the halo exchange of a sweep runs beside the sweep of the block interior
  cudaStream_t aux_stream = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  std::vector<cudaEvent_t> ev_leg;  // per sharded level: the side-stream exchange of the down leg's result
  bool overlap = true;

  ~amgb_hierarchy() {
    if (exec) cudaGraphExecDestroy(exec);
    if (graph) cudaGraphDestroy(graph);
    for (void* p : ipc_opened) cudaIpcCloseMemHandle(p);
    if (ev_fork) cudaEventDestroy(ev_fork);
    if (ev_join) cudaEventDestroy(ev_join);
    for (cudaEvent_t e : ev_leg) cudaEventDestroy(e);
    if (aux_stream) cudaStreamDestroy(aux_stream);
    if (own_stream) cudaStreamDestroy(own_stream);
    if (timed_out_host) cudaFreeHost(timed_out_host);
  }
  // Call after a stream synchronise: a halo wait that gave up means a neighbour died or stalled
  // and the vectors hold stale halos -- fail the call instead of returning them.
  void check_halo() const {
    if (timed_out_host && *(volatile int*)timed_out_host)
      throw ApiError(AMGB_ENCCL, "halo exchange timed out waiting for a neighbouring rank "
                                 "(AMGB_HALO_TIMEOUT_MS); the level vectors are invalid");
  }
  // Map the neighbours' level vectors and flag arrays into this process.
  void setup_p2p() {
    if (!comm || world() < 2 || n_sharded == 0) return;
    // highest priority: the two-block exchange kernel must be dispatched ahead of the
    // thousands of blocks of the interior sweep it overlaps with
    int prio_lo = 0, prio_hi = 0;
    CUDA_CHECK(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
    CUDA_CHECK(cudaStreamCreateWithPriority(&aux_stream, cudaStreamNonBlocking, prio_hi));
    CUDA_CHECK(cudaEventCreateWithFlags(&ev_fork, cudaEventDisableTiming));
    CUDA_CHECK(cudaEventCreateWithFlags(&ev_join, cudaEventDisableTiming));
    ev_leg.assign(n_sharded, nullptr);
    for (cudaEvent_t& e : ev_leg) CUDA_CHECK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    const char* ov = std::getenv("AMGB_OVERLAP");
    overlap = !(ov && std::string(ov) == "0");
    if (const char* tmo = std::getenv("AMGB_HALO_TIMEOUT_MS")) {
      const double ms = std::atof(tmo);
      if (ms > 0) halo_timeout_cycles = (long long)(ms * 2.0e6);  // clock64 ticks at ~2 GHz
    }
    const char* env = std::getenv("AMGB_HALO");
    if (env && std::string(env) == "nccl") return;
    const int G = world(), g = rank();
    // [site][bumped by lower / upper neighbour][arrived, data] of the stand-alone exchanges, then
    // [leg site][bumped by lower / upper neighbour] of the fused legs (struct sleg::Sync)
    // then [source rank][arrived, data] of the peer-memory all-gather
    flags.alloc((size_t)kMaxSites * 4 + (size_t)kMaxLegSites * 2 + 2 * 8);
    flags.zero(stream);
    gather_epochs.alloc(8);
    gather_epochs.zero(stream);
    gather_done.alloc(8);
    gather_done.zero(stream);
    leg_epochs.alloc((size_t)kMaxLegSites * 2);
    leg_epochs.zero(stream);
    leg_done.alloc((size_t)kMaxLegSites * 2);
    leg_done.zero(stream);
    epochs.alloc((size_t)kMaxSites * 2);
    epochs.zero(stream);
    CUDA_CHECK(cudaHostAlloc(&timed_out_host, sizeof(int), cudaHostAllocMapped));
    *timed_out_host = 0;
    CUDA_CHECK(cudaHostGetDevicePointer(&timed_out_dev, timed_out_host, 0));
    // handles: per rank [flags, then u, tmp and fw of every sharded level, then the first replicated f]
    const int per_rank = 2 + 3 * n_sharded;
    const size_t hb = sizeof(cudaIpcMemHandle_t);  // 64 bytes = 8 doubles
    std::vector<cudaIpcMemHandle_t> mine(per_rank);
    bool ok = cudaIpcGetMemHandle(&mine[0], flags.p) == cudaSuccess;
    for (int l = 0; l < n_sharded && ok; ++l) {
      ok = ok && cudaIpcGetMemHandle(&mine[1 + 3 * l], lv[l].u.p) == cudaSuccess;
      ok = ok && cudaIpcGetMemHandle(&mine[2 + 3 * l], lv[l].tmp.p) == cudaSuccess;
      ok = ok && cudaIpcGetMemHandle(&mine[3 + 3 * l], lv[l].fw.p) == cudaSuccess;
    }
    ok = ok && cudaIpcGetMemHandle(&mine[1 + 3 * n_sharded], lv[n_sharded].f.p) == cudaSuccess;
    cudaGetLastError();
    // all-gather (handles, ok flag) through NCCL on a device staging buffer
    const size_t dbl_per_rank = per_rank * hb / sizeof(double) + 1;
    DevBuf<double> stage;
    stage.alloc(dbl_per_rank * G);
    std::vector<double> host(dbl_per_rank * G, 0.0);
    std::memcpy(&host[dbl_per_rank * g], mine.data(), per_rank * hb);
    host[dbl_per_rank * g + dbl_per_rank - 1] = ok ? 1.0 : 0.0;
    CUDA_CHECK(cudaMemcpyAsync(stage.p + dbl_per_rank * g, &host[dbl_per_rank * g], dbl_per_rank * sizeof(double),
                               cudaMemcpyHostToDevice, stream));
    std::vector<int64_t> st(G + 1);
    for (int r = 0; r <= G; ++r) st[r] = (int64_t)dbl_per_rank * r;
    allgather_blocks(stage.p, st, stream);
    CUDA_CHECK(cudaMemcpyAsync(host.data(), stage.p, host.size() * sizeof(double), cudaMemcpyDeviceToHost, stream));
    CUDA_CHECK(cudaStreamSynchronize(stream));
    bool all_ok = true;
    for (int r = 0; r < G; ++r) all_ok = all_ok && host[dbl_per_rank * r + dbl_per_rank - 1] == 1.0;
    if (!all_ok) return;
    auto open = [&](int r, int idx) -> void* {
      cudaIpcMemHandle_t hnd;
      std::memcpy(&hnd, reinterpret_cast<const char*>(&host[dbl_per_rank * r]) + idx * hb, hb);
      void* p = nullptr;
      if (cudaIpcOpenMemHandle(&p, hnd, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
      }
      ipc_opened.push_back(p);
      return p;
    };
    peers.assign(n_sharded, PeerMap());
    bool mapped = true;
    if (g > 0) mapped = mapped && (peer_flags_lo = (unsigned long long*)open(g - 1, 0));
    if (g + 1 < G) mapped = mapped && (peer_flags_hi = (unsigned long long*)open(g + 1, 0));
    for (int l = 0; l < n_sharded && mapped; ++l) {
      for (int v = 0; v < 3; ++v) {
        if (g > 0) mapped = mapped && (peers[l].lo[v] = (double*)open(g - 1, 1 + 3 * l + v));
        if (g + 1 < G) mapped = mapped && (peers[l].hi[v] = (double*)open(g + 1, 1 + 3 * l + v));
      }
      if (g > 0) {
        peers[l].lo_halo_lo = plan.halo_lo[l];
        peers[l].lo_n_own = (int)(plan.start[l][g] - plan.start[l][g - 1]);
      }
    }
    // all-gather by peer-memory stores: every other rank's flags and first replicated right-hand side
    bool gmapped = mapped && G - 1 <= dev::kGatherMaxPeers && G <= 8;
    const char* gp = std::getenv("AMGB_GATHER_PUSH");
    if (gp && std::string(gp) == "0") gmapped = false;
    if (gmapped) {
      gatherp = dev::GatherParams{};
      gatherp.n_peers = G - 1;
      gatherp.src = lv[n_sharded].f.p;
      gatherp.begin = (int)coarse_block_start[g];
      gatherp.count = (int)(coarse_block_start[g + 1] - coarse_block_start[g]);
      gatherp.timed_out = timed_out_dev;
      gatherp.timeout_cycles = halo_timeout_cycles;
      const size_t goff = (size_t)kMaxSites * 4 + (size_t)kMaxLegSites * 2;
      int k = 0;
      for (int r = 0; r < G && gmapped; ++r) {
        if (r == g) continue;
        unsigned long long* pf = (r == g - 1) ? peer_flags_lo : (r == g + 1) ? peer_flags_hi : (unsigned long long*)open(r, 0);
        double* pv = (double*)open(r, 1 + 3 * n_sharded);
        gmapped = gmapped && pf && pv;
        dev::GatherPeer& R = gatherp.peer[k];
        R.dst = pv;
        R.peer_flags = pf ? pf + goff + 2 * g : nullptr;
        R.my_flags = flags.p + goff + 2 * r;
        R.epoch = gather_epochs.p + k;
        R.done = gather_done.p + k;
        ++k;
      }
    }
    // every rank must agree, otherwise some would wait for flags nobody bumps
    scalar_host_and(mapped);
    p2p = mapped;
    scalar_host_and(gmapped);
    gather_push = p2p && gmapped;
    const char* fp = std::getenv("AMGB_FUSED_PUSH");
    if (p2p && !(fp && std::string(fp) == "0")) wire_leg_sync();
  }
  // Fused halo push (stream_leg_api.hpp, struct Sync): when every sharded level runs as streaming legs,
  // each leg kernel is a site; its edge warps wait for the neighbours' previous site and push the rows
  // the neighbours keep as ghost rows straight into their vectors.  No exchange launch remains on the
  // sharded levels.
  void wire_leg_sync() {
    fused_push = false;
    const int ns = n_sharded, G = world(), g = rank();
    if (ns < 1 || 2 * ns > kMaxLegSites) return;
    for (int l = 0; l < ns; ++l)
      if (!leg_ok(l) || !legs[l].stream) return;
    const int K = 2 * ns;
    auto leg_flag = [&](unsigned long long* base, int site, int side) { return base + (size_t)kMaxSites * 4 + 2 * site + side; };
    auto wire = [&](int l, bool up) {
      sleg::Params& P = up ? legs[l].sup : legs[l].sdown;
      const LevelState& S = lv[l];
      const int site = up ? K - 1 - l : l, prev = (site + K - 1) % K;
      const int NS = sleg::stages(up ? sleg::UP : legs[l].kind_down, P.nu);
      sleg::Sync& Y = P.sync;
      Y = sleg::Sync{};
      Y.enabled = 1 | env_int("AMGB_SYNC_DEBUG", 0);  // bits 1-3 switch off wait / push / signal (timing experiments only)
      Y.timed_out = timed_out_dev;
      Y.timeout_cycles = halo_timeout_cycles;
      for (int side = 0; side < 2; ++side) {
        const bool has = side == 0 ? g > 0 : g + 1 < G;
        unsigned long long* peer_flags = side == 0 ? peer_flags_lo : peer_flags_hi;
        Y.wait_flag[side] = has ? leg_flag(flags.p, prev, side) : nullptr;
        Y.wait_epoch[side] = leg_epochs.p + 2 * prev + side;
        Y.epoch[side] = leg_epochs.p + 2 * site + side;
        Y.peer_flag[side] = has ? leg_flag(peer_flags, site, 1 - side) : nullptr;  // I am its neighbour on the other side
        Y.done[side] = leg_done.p + 2 * site + side;
      }
      // output vector: the down leg writes tmp (vector 1), the up leg u (vector 0)
      const int v = up ? 0 : 1;
      const int n_lo = (g > 0) ? (int)(plan.start[l][g] - plan.start[l][g - 1]) : 0;  // rows of rank g-1's block
      if (g > 0) {  // my first rows are rank g-1's upper ghost rows
        Y.push_u[0].dst = peers[l].lo[v] + n_lo;
        Y.push_u[0].begin = S.halo_lo;
        Y.push_u[0].end = S.halo_lo + std::min(S.halo_hi, S.n_own);
      }
      if (g + 1 < G) {  // my last rows are rank g+1's lower ghost rows
        Y.push_u[1].dst = peers[l].hi[v] - S.n_own;
        Y.push_u[1].begin = S.halo_lo + S.n_own - std::min(S.halo_lo, S.n_own);
        Y.push_u[1].end = S.halo_lo + S.n_own;
      }
      int lo_reach = P.own_begin, hi_reach = P.own_end;  // local fine rows whose producers / readers are edge warps
      if (Y.push_u[0].dst) lo_reach = std::max(lo_reach, Y.push_u[0].end);
      if (Y.push_u[1].dst) hi_reach = std::min(hi_reach, Y.push_u[1].begin);
      if (!up && l + 1 < ns) {  // the coarse right-hand side goes into the neighbours' window of level l + 1
        const LevelState& C = lv[l + 1];
        const int c_lo = (g > 0) ? (int)(plan.start[l + 1][g] - plan.start[l + 1][g - 1]) : 0;
        if (g > 0) {
          Y.push_fc[0].dst = peers[l + 1].lo[2] + c_lo;
          Y.push_fc[0].begin = C.halo_lo;
          Y.push_fc[0].end = C.halo_lo + std::min(C.halo_hi, C.n_own);
          lo_reach = std::max(lo_reach, 2 * (Y.push_fc[0].end + P.cbase) + 1 - P.base);
        }
        if (g + 1 < G) {
          Y.push_fc[1].dst = peers[l + 1].hi[2] - C.n_own;
          Y.push_fc[1].begin = C.halo_lo + C.n_own - std::min(C.halo_lo, C.n_own);
          Y.push_fc[1].end = C.halo_lo + C.n_own;
          hi_reach = std::min(hi_reach, 2 * (Y.push_fc[1].begin + P.cbase) - P.base);
        }
      }
      // edge chunks: those that read ghost rows (within NS + 2 lines of the block edge) or produce pushed rows
      sleg::classify_edges(P, NS, lo_reach, hi_reach, Y);
    };
    for (int l = 0; l < ns; ++l) {
      wire(l, false);
      wire(l, true);
    }
    fused_push = true;
  }
  // logical AND of a host bool over all ranks (NCCL all-reduce of one double)
  void scalar_host_and(bool& v) {
    double x = v ? 0.0 : 1.0;
    CUDA_CHECK(cudaMemcpyAsync(scalar.p, &x, sizeof(double), cudaMemcpyHostToDevice, stream));
    v = finish_scalar() == 0.0;
  }
  int rank() const { return comm ? comm->rank : 0; }
  int world() const { return comm ? comm->world : 1; }

  void prepare_smoother(int l) {
    if (lv[l].sharded) {
      if (opt.smoother == AMGB_SMOOTHER_GS)
        throw std::invalid_argument("lexicographic Gauss-Seidel cannot run on a sharded level");
      if (opt.smoother == AMGB_SMOOTHER_COLOR_GS) ops[l]->ensure_colors(stream);
      return;
    }
    if (opt.smoother == AMGB_SMOOTHER_GS) {
      const bool scan = opt.gs_mode == AMGB_GS_AUTO || opt.gs_mode == AMGB_GS_LINESCAN;
      if (opt.gs_mode == AMGB_GS_AUTO) ops[l]->ensure_wave(stream);
      if (scan && !ops[l]->wave_ok) ops[l]->ensure_lines(stream);
      if (!(ops[l]->wave_ok || (scan && ops[l]->lines_ok))) ops[l]->ensure_fronts(stream);
      if (!lv[l].tmp.p) lv[l].tmp.alloc(lv[l].n_vec() + 4);
    }
    if (opt.smoother == AMGB_SMOOTHER_COLOR_GS) ops[l]->ensure_colors(stream);
    if (opt.smoother == AMGB_SMOOTHER_LINE_GS) {
      ops[l]->ensure_line_gs_lines((int)m[l], opt.lines, fast_arith(), "level " + std::to_string(l), stream);
      if (!lv[l].tmp.p) lv[l].tmp.alloc(lv[l].n_vec() + 4);
    }
  }

  // Halo exchange of a halo-extended level vector with ranks g-1 / g+1: one grouped
  // NCCL send/recv pair per neighbour on the compute stream.
  void exchange(int l, double* base, cudaStream_t s) {
    const LevelState& S = lv[l];
    if (!S.sharded) return;
    NcclApi& nc = NcclApi::get();
    const int g = rank(), G = world();
    const int up_cnt = plan.halo_hi[l];  // what rank g-1 keeps above its block = my first rows
    const int dn_cnt = plan.halo_lo[l];  // what rank g+1 keeps below its block = my last rows
    ++halo_exchanges_per_vcycle;
    if (p2p) {
      const int v = (base == S.u.p) ? 0 : (base == S.tmp.p ? 1 : 2);
      // flags and epochs are per site, epochs only ever grow: a site may be reused (every rank makes the
      // same sequence of exchanges, so they all wrap at the same call)
      const int site = site_cursor++ % kMaxSites;
      dev::HaloSide lo{}, hi{};
      if (g > 0) {  // my first rows -> rank g-1's upper halo
        lo.peer_dst = peers[l].lo[v] + peers[l].lo_halo_lo + peers[l].lo_n_own;
        lo.src = base + S.halo_lo;
        lo.count = up_cnt;
        lo.peer_flag = peer_flags_lo + 4 * site + 2;  // "bumped by your upper neighbour"
        lo.my_flag = flags.p + 4 * site + 0;
      }
      if (g + 1 < G) {  // my last rows -> rank g+1's lower halo
        hi.peer_dst = peers[l].hi[v];
        hi.src = base + S.halo_lo + S.n_own - dn_cnt;
        hi.count = dn_cnt;
        hi.peer_flag = peer_flags_hi + 4 * site + 0;  // "bumped by your lower neighbour"
        hi.my_flag = flags.p + 4 * site + 2;
      }
      LAUNCH(dev::k_halo_exchange, 2, 1024, 0, s, lo, hi, epochs.p + 2 * site, timed_out_dev, halo_timeout_cycles);
      return;
    }
    NCCL_CHECK(nc.GroupStart());
    if (g > 0) {
      NCCL_CHECK(nc.Send(base + S.halo_lo, up_cnt, ncclDouble, g - 1, comm->comm, s));
      NCCL_CHECK(nc.Recv(base, S.halo_lo, ncclDouble, g - 1, comm->comm, s));
    }
    if (g + 1 < G) {
      NCCL_CHECK(nc.Send(base + S.halo_lo + S.n_own - dn_cnt, dn_cnt, ncclDouble, g + 1, comm->comm, s));
      NCCL_CHECK(nc.Recv(base + S.halo_lo + S.n_own, S.halo_hi, ncclDouble, g + 1, comm->comm, s));
    }
    NCCL_CHECK(nc.GroupEnd());
  }
  // the first replicated right-hand side: every rank gets the blocks the other ranks produced
  void gather_coarse_rhs(cudaStream_t s) {
    if (gather_push) {
      LAUNCH(dev::k_allgather_push, gatherp.n_peers * dev::kGatherSlices, 512, 0, s, gatherp);
      return;
    }
    allgather_blocks(lv[n_sharded].f.p, coarse_block_start, s);
  }
  // every rank contributes its block [start[r], start[r+1]) of a full-length vector
  void allgather_blocks(double* full, const std::vector<int64_t>& start, cudaStream_t s) {
    NcclApi& nc = NcclApi::get();
    NCCL_CHECK(nc.GroupStart());
    for (int r = 0; r < world(); ++r) {
      const int64_t cnt = start[r + 1] - start[r];
      if (cnt > 0)
        NCCL_CHECK(nc.Broadcast(full + start[r], full + start[r], (size_t)cnt, ncclDouble, r, comm->comm, s));
    }
    NCCL_CHECK(nc.GroupEnd());
  }

  // One damped-Jacobi sweep src -> dst of level l (halo-extended vectors); on a sharded level the halo
  // exchange with ranks +-1 runs on the side stream beside the sweep of the block interior.
  void jacobi_sweep(int l, double* src, double* dst, cudaStream_t s) {
    Operator& A = *ops[l];
    LevelState& S = lv[l];
    const int w = S.halo_lo;  // >= half-bandwidth: rows [w, n_own - w) read no halo entry
    if (S.sharded && overlap && aux_stream && S.n_own > 4 * w) {
      CUDA_CHECK(cudaEventRecord(ev_fork, s));
      CUDA_CHECK(cudaStreamWaitEvent(aux_stream, ev_fork, 0));
      exchange(l, src, aux_stream);  // enqueued first, on the high-priority stream
      A.jacobi_rows(src + S.halo_lo, S.f.p, opt.omega, dst + S.halo_lo, w, S.n_own - w, s);
      CUDA_CHECK(cudaEventRecord(ev_join, aux_stream));
      CUDA_CHECK(cudaStreamWaitEvent(s, ev_join, 0));
      A.jacobi_edges(src + S.halo_lo, S.f.p, opt.omega, dst + S.halo_lo, w, w, s);
    } else {
      exchange(l, src, s);
      A.jacobi(src + S.halo_lo, S.f.p, opt.omega, dst + S.halo_lo, s);
    }
  }
  // smoother->smooth(A_l, u_l, f_l)   (multigrid.hpp:268-269, :300-301)
  // from_zero:   u_l is known to be zero (pre-smoothing of a coarse level, :278)
  // with_prolong: the coarse-grid correction u_l += P u_{l+1} (:294-296) has not been applied
  //               yet and is folded into the first sweep (Jacobi) or applied first (others)
  void smooth(int l, cudaStream_t s, bool from_zero = false, bool with_prolong = false) {
    Operator& A = *ops[l];
    LevelState& S = lv[l];
    const int64_t iters = opt.smoother_iters;
    if (opt.smoother != AMGB_SMOOTHER_JACOBI || iters < 1) {
      if (with_prolong) prolong_add(l, s);
      if (opt.smoother == AMGB_SMOOTHER_GS) {
        for (int64_t it = 0; it < iters; ++it) {  // smoother.hpp:195-198
          A.gs_direction(true, S.f.p, S.u.p, S.tmp.p, opt.gs_mode, s);
          A.gs_direction(false, S.f.p, S.u.p, S.tmp.p, opt.gs_mode, s);
        }
      } else if (opt.smoother == AMGB_SMOOTHER_LINE_GS) {
        for (int64_t it = 0; it < iters; ++it) {
          A.line_gs_half(true, opt.lines, fast_arith(), S.f.p, S.u.p, S.tmp.p, s);
          A.line_gs_half(false, opt.lines, fast_arith(), S.f.p, S.u.p, S.tmp.p, s);
        }
      } else if (opt.smoother == AMGB_SMOOTHER_COLOR_GS) {
        // Row-block sharded level: the colour mirrors list global rows, so the vectors are handed over
        // shifted to global numbering; one halo exchange before every colour pass (a pass reads the
        // other colours' latest values, some of which live on ranks +-1).
        double* u_g = S.sharded ? S.u.p - (S.s - S.halo_lo) : S.u.p;
        const double* f_g = S.sharded ? S.f.p - S.s : S.f.p;
        for (int64_t it = 0; it < iters; ++it) {
          for (int c = 0; c < A.n_colors; ++c) {
            exchange(l, S.u.p, s);
            A.color_pass(c, f_g, u_g, s);
          }
          for (int c = A.n_colors - 1; c >= 0; --c) {
            exchange(l, S.u.p, s);
            A.color_pass(c, f_g, u_g, s);
          }
        }
      }
      return;
    }
    double* src = S.u.p;
    double* dst = S.tmp.p;
    for (int64_t it = 0; it < iters; ++it) {
      bool done = false;
      if (it == 0 && from_zero && (opt.fuse & 1)) {
        done = A.jacobi_from_zero(S.f.p, opt.omega, dst + S.halo_lo, s);
      } else if (it == 0 && with_prolong && (opt.fuse & 2)) {
        // u_l's halos are still current (u_l has not changed since the down-leg exchange);
        // the coarse halos are exchanged here
        LevelState& C = lv[l + 1];
        if (C.sharded) exchange(l + 1, C.u.p, s);
        const int e_first = C.sharded ? (int)(C.s - C.halo_lo) : 0;
        A.jacobi_prolong(src + S.halo_lo, C.u.p, e_first, (int)n[l + 1], (int)S.s, S.f.p, opt.omega,
                         dst + S.halo_lo, s);
        done = true;
      }
      if (!done) {
        if (it == 0 && with_prolong) prolong_add(l, s);
        jacobi_sweep(l, src, dst, s);
      }
      std::swap(src, dst);
    }
    if (src != S.u.p)
      CUDA_CHECK(cudaMemcpyAsync(S.u_own(), src + S.halo_lo, sizeof(double) * S.n_own,
                                 cudaMemcpyDeviceToDevice, s));
  }
  // f_{l+1} = R_l (f_l - A_l u_l), u_{l+1} = 0   (multigrid.hpp:272-282)
  void residual_restrict(int l, cudaStream_t s) {
    LevelState& F = lv[l];
    LevelState& C = lv[l + 1];
    if (sa()) {  // residual into the level's scratch vector, then the restriction (transfer_sa.cuh)
      ops[l]->residual(F.u.p, F.f.p, F.tmp.p, s);
      restrict_sa(F.tmp.p, C.f.p, C.u.p, l, s);
      return;
    }
    if (bilinear()) {
      const int m_h = (int)m[l], m_H = (int)m[l + 1];
      if (!F.sharded) {
        ops[l]->residual_restrict2d(F.u.p, F.f.p, m_h, 0, C.f.p, C.u.p, m_H, 0, 0, m_H, s);
        return;
      }
      // the block's own coarse lines (and the coarse ghost lines above them when the coarse level is
      // sharded too) restrict from the own and ghost fine lines, whose residual this rank forms itself
      exchange(l, F.u.p, s);
      CUDA_CHECK(cudaMemsetAsync(C.u.p, 0, sizeof(double) * C.u.n, s));
      const int y0 = (int)(F.s / m_h);
      if (C.sharded) {
        const int Y0 = (int)(C.s / m_H);
        ops[l]->residual_restrict2d(F.u_own(), F.f.p, m_h, y0, C.f.p, C.u_own(), m_H, Y0, Y0, Y0 + C.n_mat / m_H, s);
      } else {
        const std::vector<int64_t>& cs = coarse_block_start;
        ops[l]->residual_restrict2d(F.u_own(), F.f.p, m_h, y0, C.f.p, C.u.p, m_H, 0, (int)(cs[rank()] / m_H),
                                    (int)(cs[rank() + 1] / m_H), s);
        gather_coarse_rhs(s);
      }
      return;
    }
    if (!F.sharded) {
      ops[l]->residual_restrict(F.u.p, F.f.p, C.f.p, C.u.p, (int)n[l + 1], s);
      return;
    }
    exchange(l, F.u.p, s);
    CUDA_CHECK(cudaMemsetAsync(C.u.p, 0, sizeof(double) * C.u.n, s));
    if (C.sharded) {
      ops[l]->residual_restrict(F.u_own(), F.f.p, C.f.p, C.u_own(), C.n_mat, s);
    } else {
      // first agglomerated level: every rank writes its coarse block straight into the
      // full-length rhs, then the blocks are exchanged so each rank holds a replica
      const std::vector<int64_t>& cs = coarse_block_start;
      const int64_t c0 = cs[rank()], c1 = cs[rank() + 1];
      ops[l]->residual_restrict(F.u_own(), F.f.p, C.f.p + c0, C.u.p + c0, (int)(c1 - c0), s);
      gather_coarse_rhs(s);
    }
  }
  // u_l = u_l + P_l u_{l+1}   (multigrid.hpp:294-296)
  void prolong_add(int l, cudaStream_t s) {
    LevelState& F = lv[l];
    LevelState& C = lv[l + 1];
    if (sa()) {
      prolong_add_sa(C.u.p, F.u.p, l, s);
      return;
    }
    if (bilinear()) {
      if (!F.sharded) {
        prolong_add2d(C.u.p, F.u.p, l, s);
        return;
      }
      // the first fine line of the block reads the coarse line below the coarse block (coarse halo)
      if (C.sharded) exchange(l + 1, C.u.p, s);
      const int m_h = (int)m[l], m_H = (int)m[l + 1];
      const int y0 = (int)(F.s / m_h), y1 = (int)(F.e / m_h);
      const double* e = C.sharded ? C.u_own() : C.u.p;
      const int Y_first = C.sharded ? (int)(C.s / m_H) : 0;
      LAUNCH(dev::k_prolong_add2d, dim3(blocks_for(m_h, 256), (unsigned)blocks_for(y1 - y0, 2)), 256, 0, s, e, m_H,
             Y_first, F.u_own(), m_h, y0, y0, y1);
      return;
    }
    if (C.sharded) exchange(l + 1, C.u.p, s);  // needs e[s_c - 1]
    const int e_first = C.sharded ? (int)(C.s - C.halo_lo) : 0;
    if ((reinterpret_cast<uintptr_t>(F.u_own()) & 15) == 0 && (F.s & 1) == 0)
      LAUNCH(dev::k_prolong_add2, blocks_for((F.n_own + 1) / 2, 256), 256, 0, s, C.u.p, e_first, (int)n[l + 1],
             F.u_own(), (int)F.s, F.n_own);
    else
      LAUNCH(dev::k_prolong_add, blocks_for(F.n_own, 256), 256, 0, s, C.u.p, e_first, (int)n[l + 1],
             F.u_own(), (int)F.s, F.n_own);
  }
  // u_l += P_l e on a 2-D hierarchy (e: m_{l+1}^2 coarse values, u: m_l^2 fine values)
  void prolong_add2d(const double* e, double* u, int l, cudaStream_t s) const {
    if (m[l] < 1) return;
    LAUNCH(dev::k_prolong_add2d, dim3(blocks_for(m[l], 256), (unsigned)blocks_for(m[l], 2)), 256, 0, s, e, (int)m[l + 1], 0,
           u, (int)m[l], 0, 0, (int)m[l]);
  }
  // f_c = R_l r on a 2-D hierarchy
  void restrict2d(const double* r, double* f_c, int l, cudaStream_t s) const {
    if (m[l + 1] < 1) return;
    LAUNCH(dev::k_restrict2d, dim3(blocks_for(m[l + 1], 256), (unsigned)m[l + 1]), 256, 0, s, r, (int)m[l], f_c,
           (int)m[l + 1]);
  }
  // f_c = R_l r (and u_c = 0 unless u_c is null) on a smoothed-aggregation hierarchy
  void restrict_sa(const double* r, double* f_c, double* u_c, int l, cudaStream_t s) const {
    const DevSell& R = sa_R_rows[l];
    if (R.n_rows < 1) return;
    if (fast_arith()) LAUNCH(sa::k_restrict_sa<true>, blocks_for(R.n_rows, 256), 256, 0, s, R.view(), r, f_c, u_c);
    else LAUNCH(sa::k_restrict_sa<false>, blocks_for(R.n_rows, 256), 256, 0, s, R.view(), r, f_c, u_c);
  }
  // u_l += P_l e on a smoothed-aggregation hierarchy
  void prolong_add_sa(const double* e, double* u, int l, cudaStream_t s) const {
    const DevSell& P = sa_P_rows[l];
    if (P.n_rows < 1) return;
    if (fast_arith()) LAUNCH(sa::k_prolong_add_sa<true>, blocks_for(P.n_rows, 256), 256, 0, s, P.view(), e, u);
    else LAUNCH(sa::k_prolong_add_sa<false>, blocks_for(P.n_rows, 256), 256, 0, s, P.view(), e, u);
  }
  // P_l of this hierarchy's transfer kind (host setup)
  Csc prolongation(int l) const {
    if (sa()) return sa_resident ? sa_dev_P[l].download(stream) : sa_P[l];
    return bilinear() ? make_prolongation_2d(m[l], m[l + 1]) : make_prolongation(n[l], n[l + 1]);
  }
  void coarse_solve(cudaStream_t s) {  // multigrid.hpp:287-288
    const int nc = factor.n, bw = factor.bw;
    int threads = std::min(1024, std::max(32, ((bw + 31) / 32) * 32));
    const size_t xbytes = sizeof(double) * (size_t)nc;
    const size_t lbytes = sizeof(double) * (size_t)nc * std::max(bw, 1);
    const size_t cap = 200 * 1024;
    if (bw >= 1 && bw <= 8 && xbytes + lbytes <= 48 * 1024) {
      LAUNCH(dev::k_banded_ldlt_solve_serial, 1, 128, xbytes + lbytes, s, dL.p, dd.p, nc, bw, lv[L - 1].f.p,
             lv[L - 1].u.p);
      return;
    }
    if (bw <= 31 && xbytes <= cap) {
      const int l_smem = xbytes + lbytes <= cap;
      const size_t smem = xbytes + (l_smem ? lbytes : 0);
      if (smem > 48 * 1024 && !ldlt_warp_attr_set) {
        CUDA_CHECK(cudaFuncSetAttribute(dev::k_banded_ldlt_solve_warp,
                                        cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cap));
        ldlt_warp_attr_set = true;
      }
      LAUNCH(dev::k_banded_ldlt_solve_warp, 1, 32, smem, s, dL.p, dd.p, nc, bw, lv[L - 1].f.p, lv[L - 1].u.p,
             l_smem);
      return;
    }
    const int x_smem = xbytes <= cap;
    const int l_smem = x_smem && xbytes + lbytes <= cap;
    const size_t smem = (x_smem ? xbytes : 0) + (l_smem ? lbytes : 0);
    if (smem > 48 * 1024 && !ldlt_attr_set) {
      CUDA_CHECK(cudaFuncSetAttribute(dev::k_banded_ldlt_solve, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)cap));
      ldlt_attr_set = true;
    }
    LAUNCH(dev::k_banded_ldlt_solve, 1, threads, smem, s, dL.p, dd.p, nc, bw, lv[L - 1].f.p, lv[L - 1].u.p,
           dwork.p, x_smem, l_smem);
  }
  std::vector<int64_t> coarse_block_start;  // block starts of level n_sharded (image of the fine blocks)

  // ---- fused legs (fused_leg.cuh): one kernel per level and leg of the damped-Jacobi cycle
  struct LegLevel {
    bool ok = false;
    bool stream = false;      // true: stream_leg.cuh (registers + shuffles); false: fused_leg.cuh (TMA rings)
    leg::Plan down, up;
    sleg::Params sdown{}, sup{};
    unsigned mask = 0;
    int kind_down = 0;
    bool matrix_free = false;  // the level's operator was verified to be a constant five-point stencil
    bool half = false;         // the level's operator was verified to be bitwise symmetric: legs stream its upper half
    // row-type dictionary (option fuse bit 7): one byte per row + the table of the level's distinct rows
    int dict_types = 0;
    DevBuf<unsigned char> tid;
    DevBuf<double> table;
  };
  std::vector<LegLevel> legs;
  static int env_int(const char* name, int dflt) {
    const char* v = std::getenv(name);
    return v ? std::atoi(v) : dflt;
  }
  template <int ND, int NS>
  static void leg_attr() {
    CUDA_CHECK(cudaFuncSetAttribute(leg::k_fused_leg<ND, NS>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    227 * 1024));
    CUDA_CHECK(cudaFuncSetAttribute(leg::k_fused_leg<ND, NS>, cudaFuncAttributePreferredSharedMemoryCarveout,
                                    cudaSharedmemCarveoutMaxShared));
  }
  template <int ND, int NS>
  static void leg_launch(const leg::Plan& pl, cudaStream_t s) {
    auto kern = leg::k_fused_leg<ND, NS>;
    LAUNCH(kern, pl.tiles, pl.threads, pl.smem_bytes, s, pl.P);
  }
  // action 0: opt the instantiation in to large dynamic shared memory; 1: launch
  static void leg_dispatch(const leg::Plan& pl, int action, cudaStream_t s) {
    auto go = [&](auto nd_tag) {
      constexpr int ND = decltype(nd_tag)::value;
      switch (pl.P.NS) {
        case 1: action ? leg_launch<ND, 1>(pl, s) : leg_attr<ND, 1>(); break;
        case 2: action ? leg_launch<ND, 2>(pl, s) : leg_attr<ND, 2>(); break;
        case 3: action ? leg_launch<ND, 3>(pl, s) : leg_attr<ND, 3>(); break;
        default: throw ApiError(AMGB_ESTATE, "fused leg: unsupported stage count");
      }
    };
    if (pl.P.nd <= 6) go(std::integral_constant<int, 6>());
    else go(std::integral_constant<int, 10>());
  }
  // ---- register-streaming legs (stream_leg.cuh, compiled in legs.cu)
  bool fast_arith() const { return opt.arith == AMGB_ARITH_FAST; }
  bool sleg_dispatch(int kind, unsigned mask, const sleg::Params& P, cudaStream_t s, int action,
                     int* wps = nullptr) const {
    const bool done = sleg::dispatch(kind, mask, P, s, action, wps, fast_arith());
    if (done && action == 1) g_launches.fetch_add(1, std::memory_order_relaxed);
    return done;
  }
  // Matrix-free legs (option fuse bit 6): true when the mirror D (row t = global row base + t) is bit
  // for bit the constant five-point stencil cst[] on the offsets -m, -1, 0, +1, +m (setup_dia.cuh).
  bool check_matrix_free(const DevDia& D, int base, int n_global, int m, double (&cst)[5]) {
    if (!(opt.fuse & 64) || D.n_diag != 5 || m < 3 || n_global < 3 * m) return false;
    const int want[5] = {-m, -1, 0, 1, m};
    for (int d = 0; d < 5; ++d)
      if (D.off[d] != want[d]) return false;
    // an interior row of the mirror gives the five coefficients
    int64_t kg = std::max<int64_t>(base, 0);
    kg = (kg / m + 1) * (int64_t)m + 1;
    const int64_t t0 = kg - base;
    if (t0 < 0 || t0 >= D.n_rows || kg >= (int64_t)n_global - m - 1) return false;
    setup::Const5 C{};
    for (int d = 0; d < 5; ++d)
      CUDA_CHECK(cudaMemcpyAsync(&C.c[d], D.val.p + (size_t)d * D.ld + t0, sizeof(double), cudaMemcpyDeviceToHost, stream));
    CUDA_CHECK(cudaStreamSynchronize(stream));
    for (int d = 0; d < 5; ++d)
      if (C.c[d] == 0.0) return false;
    DevBuf<int> bad;
    bad.alloc(1);
    bad.zero(stream);
    LAUNCH(setup::k_check_const5, blocks_for(D.n_rows, 256), 256, 0, stream, D.val.p, D.n_rows, D.ld, base, n_global, m, C,
           bad.p);
    int hb = 1;
    CUDA_CHECK(cudaMemcpyAsync(&hb, bad.p, sizeof(int), cudaMemcpyDeviceToHost, stream));
    CUDA_CHECK(cudaStreamSynchronize(stream));
    if (hb) return false;
    for (int d = 0; d < 5; ++d) cst[d] = C.c[d];
    return true;
  }
  // Half-streaming legs: true when the square DIA mirror D is bitwise symmetric, A(r, r+o) == A(r+o, r) for
  // every stored entry, and stores nothing outside the level (setup_dia.cuh)
  bool check_symmetric(const DevDia& D) {
    if (D.n_rows < 1 || D.n_diag < 1 || D.n_diag > setup::kMaxOffsets) return false;
    setup::Offsets off{};
    off.n = D.n_diag;
    for (int d = 0; d < D.n_diag; ++d) off.v[d] = D.off[d];
    DevBuf<int> flag;
    flag.alloc(1);
    flag.zero(stream);
    LAUNCH(setup::k_dia_asymmetric, blocks_for(D.n_rows, 256), 256, 0, stream, D.val.p, D.n_rows, D.ld, off, flag.p);
    int asym = 1;
    CUDA_CHECK(cudaMemcpyAsync(&asym, flag.p, sizeof(int), cudaMemcpyDeviceToHost, stream));
    CUDA_CHECK(cudaStreamSynchronize(stream));
    return asym == 0;
  }
  // Row-type dictionary of a DIA mirror (option fuse bit 7): at most 256 distinct rows, every row
  // verified bit for bit against its table row.  Returns the number of types (0: not applicable).
  int build_dictionary(const DevDia& D, DevBuf<unsigned char>& tid, DevBuf<double>& table) {
    if (!(opt.fuse & 128) || D.n_rows < 1 || D.n_diag < 1) return 0;
    cudaStream_t s = stream;
    const int n = D.n_rows, nd = D.n_diag;
    DevBuf<unsigned long long> keys;
    keys.alloc(setup::kDictSlots);
    keys.zero(s);
    DevBuf<int> rep, flag;
    std::vector<int> hrep(setup::kDictSlots, 0x7fffffff);
    rep.upload(hrep, s);
    flag.alloc(1);
    flag.zero(s);
    LAUNCH(setup::k_dict_insert, blocks_for(n, 256), 256, 0, s, D.val.p, n, D.ld, nd, keys.p, rep.p, flag.p);
    int hflag = 0;
    CUDA_CHECK(cudaMemcpyAsync(hrep.data(), rep.p, hrep.size() * sizeof(int), cudaMemcpyDeviceToHost, s));
    CUDA_CHECK(cudaMemcpyAsync(&hflag, flag.p, sizeof(int), cudaMemcpyDeviceToHost, s));
    CUDA_CHECK(cudaStreamSynchronize(s));
    if (hflag) return 0;
    std::vector<std::pair<int, int>> used;  // (representative row, slot): ids in order of first appearance
    for (int k = 0; k < setup::kDictSlots; ++k)
      if (hrep[k] != 0x7fffffff) used.emplace_back(hrep[k], k);
    if (used.empty() || used.size() > 256) return 0;
    std::sort(used.begin(), used.end());
    std::vector<short> slot_id(setup::kDictSlots, -1);
    std::vector<int> rep_of_id(used.size());
    for (size_t i = 0; i < used.size(); ++i) {
      slot_id[used[i].second] = (short)i;
      rep_of_id[i] = used[i].first;
    }
    const int T = (int)used.size();
    DevBuf<short> d_slot_id;
    d_slot_id.upload(slot_id, s);
    DevBuf<int> d_rep;
    d_rep.upload(rep_of_id, s);
    table.alloc((size_t)T * nd);
    tid.alloc((size_t)n + 8);
    tid.zero(s);
    LAUNCH(setup::k_dict_table, blocks_for(T * nd, 256), 256, 0, s, D.val.p, D.ld, nd, d_rep.p, T, table.p);
    flag.zero(s);
    LAUNCH(setup::k_dict_assign, blocks_for(n, 256), 256, 0, s, D.val.p, n, D.ld, nd, keys.p, d_slot_id.p, table.p, tid.p,
           flag.p);
    CUDA_CHECK(cudaMemcpyAsync(&hflag, flag.p, sizeof(int), cudaMemcpyDeviceToHost, s));
    CUDA_CHECK(cudaStreamSynchronize(s));
    if (hflag) {
      table.release();
      tid.release();
      return 0;
    }
    return T;
  }
  void leg_down(int l, cudaStream_t s) {
    const LegLevel& G = legs[l];
    if (G.stream) sleg_dispatch(G.kind_down, G.mask, G.sdown, s, 1);
    else leg_dispatch(G.down, 1, s);
  }
  void leg_up(int l, cudaStream_t s) {
    const LegLevel& G = legs[l];
    if (G.stream) sleg_dispatch(sleg::UP, G.mask, G.sup, s, 1);
    else leg_dispatch(G.up, 1, s);
  }
  // Plan the fused legs of level l (whole levels of a damped-Jacobi cycle with a banded DIA
  // operator); levels the plan does not cover keep the per-operator kernels.
  //   fuse bit 2: register-streaming legs for 3 x 3 line stencils (one or two sweeps per smooth call)
  //   fuse bit 3: TMA-ring legs for the other banded levels
  void prepare_legs(int l) {
    if ((int)legs.size() != L) {
      legs.clear();
      legs.resize(L);
    }
    if ((int)leg_side.size() != L) leg_side.assign(L, 0);
    LegLevel& G = legs[l];
    G.ok = false;
    G.half = false;
    if (!(opt.fuse & 12) || opt.smoother != AMGB_SMOOTHER_JACOBI || opt.smoother_iters < 1 || l + 1 >= L) return;
    const LevelState& S = lv[l];
    if (!S.tmp.p) return;
    const int kind_down = (l == 0) ? leg::DOWN_U : leg::DOWN_ZERO;
    const int nu = (int)opt.smoother_iters;
    G.kind_down = kind_down;
    if (S.sharded) {
      // row block + ghost rows: the streaming kernels run on the rank's window of the level
      const DevDia& W = ops[l]->win;
      if (!(opt.fuse & 4) || (nu != 1 && nu != 2) || !W.val.p || W.n_diag > 10) return;
      leg::Plan st = leg::plan_leg(leg::UP, nu, (int)n[l], W.n_diag, ops[l]->win_off.data(), 148, 200 * 1024);
      if (!st.ok || !(st.P.m < st.P.n) || st.P.rho != 1) return;
      int wmax = 0;
      for (int o : ops[l]->win_off) wmax = std::max(wmax, std::abs(o));
      // three chained stencil stages + the restriction's neighbours reach 3 wmax + 1 rows out
      if (S.halo_lo < 3 * wmax + 4 || S.halo_hi < 3 * wmax + 4) return;  // ghost zone too thin
      unsigned mask = 0;
      for (int d = 0; d < W.n_diag; ++d) mask |= 1u << ((st.P.line_a[d] + 1) * 3 + st.P.delta[d] + 1);
      sleg::Params dummy{};
      dummy.nu = nu;
      if (!sleg_dispatch(kind_down, mask, dummy, nullptr, 0) || !sleg_dispatch(sleg::UP, mask, dummy, nullptr, 0)) return;
      int n_sm = 148;
      CUDA_CHECK(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, device));
      const LevelState& C = lv[l + 1];
      double cst[5] = {0, 0, 0, 0, 0};
      const bool mf = mask == sleg::kMask5 && check_matrix_free(W, (int)(S.s - S.halo_lo), (int)n[l], st.P.m, cst);
      dummy.matrix_free = mf;
      G.matrix_free = mf;
      G.dict_types = mf ? 0 : build_dictionary(W, G.tid, G.table);
      dummy.dict_types = G.dict_types;
      auto plan = [&](int kind, int NS, int X) {
        int wps = 12;
        sleg_dispatch(kind, mask, dummy, nullptr, 2, &wps);
        const int warps_target = n_sm * env_int("AMGB_SLEG_WARPS_PER_SM", wps);
        sleg::Params P{};
        P.dict_types = G.dict_types;
        P.tid = G.tid.p;
        P.table = G.table.p;
        P.nu = nu;
        P.base = (int)(S.s - S.halo_lo);
        P.n_global = (int)n[l];
        P.own_begin = S.halo_lo;
        P.own_end = S.halo_lo + S.n_own;
        P.cbase = C.sharded ? (int)(C.s - C.halo_lo) : 0;
        P.n_e = C.sharded ? (int)C.n_vec() : (int)n[l + 1];
        P.n = (int)S.n_vec();
        P.m = st.P.m;
        P.n_lines = (P.n + P.m - 1) / P.m;
        P.Wu = 32 - 2 * (NS + X);
        P.n_strips = (P.m + P.Wu - 1) / P.Wu;
        const int chunks = std::max(1, std::min(warps_target / P.n_strips, P.n_lines / env_int("AMGB_SLEG_MINLINES", 8)));
        P.set_chunks(chunks, env_int("AMGB_SLEG_EDGE_HALF", 1) != 0);  // (only used with the fused halo push)
        P.ld = W.ld;
        P.n_coarse = (int)n[l + 1];
        P.omega = opt.omega;
        P.val = W.val.p;
        P.f = S.fw.p;
        // L2 prefetch two lines beyond the register ring pays on the HBM-bound levels (measured:
        // level 0 down leg 231 -> 197 us, profiles/r2_stream_legs.md) and costs issue slots below
        P.l2_ahead = env_int("AMGB_SLEG_L2AHEAD", S.n_vec() >= (1 << 21) ? 2 : 0);
        P.matrix_free = mf;
        for (int d = 0; d < 5; ++d) P.cst[d] = cst[d];
        P.finish(W.n_diag);
        return P;
      };
      G.sdown = plan(kind_down, kind_down == leg::DOWN_U ? nu + 1 : nu, 1);
      G.sdown.uin = S.u.p;
      G.sdown.uout = S.tmp.p;
      G.sdown.fc = C.sharded ? C.fw.p : C.f.p;
      G.sup = plan(sleg::UP, nu, 0);
      G.sup.uin = S.tmp.p;
      G.sup.e = C.u.p;
      G.sup.uout = S.u.p;
      G.mask = mask;
      G.stream = true;
      G.ok = true;
      return;
    }
    const DevMat& A = ops[l]->rows_of_A();
    if (!A.is_dia || A.dia.n_diag > 10 || A.dia.rows.p) return;
    if ((opt.fuse & 4) && (nu == 1 || nu == 2)) {
      // line structure from the TMA-ring planner; the streaming kernels need rho == 1
      leg::Plan st = leg::plan_leg(leg::UP, nu, (int)n[l], A.dia.n_diag, A.dia.off, 148, 200 * 1024);
      if (st.ok && st.P.m < st.P.n && st.P.rho == 1) {
        unsigned mask = 0;
        for (int d = 0; d < A.dia.n_diag; ++d) mask |= 1u << ((st.P.line_a[d] + 1) * 3 + st.P.delta[d] + 1);
        sleg::Params dummy{};
        dummy.nu = nu;
        if (sleg_dispatch(kind_down, mask, dummy, nullptr, 0) && sleg_dispatch(sleg::UP, mask, dummy, nullptr, 0)) {
          int n_sm = 148;
          CUDA_CHECK(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, device));
          double cst[5] = {0, 0, 0, 0, 0};
          const bool mf = mask == sleg::kMask5 && check_matrix_free(A.dia, 0, (int)n[l], st.P.m, cst);
          dummy.matrix_free = mf;
          G.matrix_free = mf;
          G.dict_types = mf ? 0 : build_dictionary(A.dia, G.tid, G.table);
          dummy.dict_types = G.dict_types;
          // sharded levels (branch above) stream every diagonal: their ghost rows would need one more operator line
          G.half = !mf && G.dict_types == 0 && check_symmetric(A.dia);
          dummy.half = G.half;
          auto plan = [&](int kind, int NS, int X) {
            int wps = 12;
            sleg_dispatch(kind, mask, dummy, nullptr, 2, &wps);
            const int warps_target = n_sm * env_int("AMGB_SLEG_WARPS_PER_SM", wps);
            sleg::Params P{};
            P.dict_types = G.dict_types;
            P.tid = G.tid.p;
            P.table = G.table.p;
            P.nu = nu;
            P.base = 0;
            P.n_global = (int)n[l];
            P.own_begin = 0;
            P.own_end = (int)n[l];
            P.cbase = 0;
            P.n_e = (int)n[l + 1];
            P.n = (int)n[l];
            P.m = st.P.m;
            P.n_lines = st.P.n_lines;
            P.Wu = 32 - 2 * (NS + X);
            P.n_strips = (P.m + P.Wu - 1) / P.Wu;
            const int chunks = std::max(1, std::min(warps_target / P.n_strips, P.n_lines / env_int("AMGB_SLEG_MINLINES", 8)));
            P.set_chunks(chunks, false);
            P.ld = A.dia.ld;
            P.n_coarse = (int)n[l + 1];
            P.omega = opt.omega;
            P.val = A.dia.val.p;
            P.f = S.f.p;
            // L2 prefetch two lines beyond the register ring pays on the HBM-bound levels (measured:
            // level 0 down leg 231 -> 197 us, profiles/r2_stream_legs.md) and costs issue slots below
            P.l2_ahead = env_int("AMGB_SLEG_L2AHEAD", n[l] >= (1 << 21) ? 2 : 0);
            P.matrix_free = mf;
            P.half = G.half;
            for (int d = 0; d < 5; ++d) P.cst[d] = cst[d];
            P.finish(A.dia.n_diag);
            return P;
          };
          G.sdown = plan(kind_down, kind_down == leg::DOWN_U ? nu + 1 : nu, 1);
          G.sdown.uin = S.u.p;
          G.sdown.uout = S.tmp.p;
          G.sdown.fc = lv[l + 1].f.p;
          G.sup = plan(sleg::UP, nu, 0);
          G.sup.uin = S.tmp.p;
          G.sup.e = lv[l + 1].u.p;
          G.sup.uout = S.u.p;
          G.mask = mask;
          G.stream = true;
          G.ok = true;
          return;
        }
      }
    }
    if (!(opt.fuse & 8)) return;
    if ((kind_down == leg::DOWN_U ? nu + 1 : nu) > 3 || nu > 3) return;
    int n_sm = 148;
    CUDA_CHECK(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, device));
    const int W_ovr = env_int("AMGB_LEG_W", 0), LJ_ovr = env_int("AMGB_LEG_LJ", 0), PF_ovr = env_int("AMGB_LEG_PF", 0);
    const int occ_want = env_int("AMGB_LEG_OCC", 2);
    auto plan = [&](int kind) {
      leg::Plan pl;
      for (int occ = occ_want; occ >= 1; --occ) {
        const size_t cap = (size_t)(227 * 1024) / occ - (occ > 1 ? 1024 : 0);
        pl = leg::plan_leg(kind, nu, (int)n[l], A.dia.n_diag, A.dia.off, n_sm * occ, cap, W_ovr, LJ_ovr, PF_ovr);
        if (pl.ok && (occ == 1 || pl.P.W >= std::min(pl.P.m, 6 * pl.P.H))) break;
      }
      return pl;
    };
    G.down = plan(kind_down);
    G.up = plan(leg::UP);
    if (!G.down.ok || !G.up.ok) return;
    auto fill = [&](leg::Plan& pl) {
      pl.P.ld = A.dia.ld;
      pl.P.val = A.dia.val.p;
      pl.P.f = S.f.p;
      pl.P.omega = opt.omega;
      pl.P.n_coarse = (int)n[l + 1];
    };
    fill(G.down);
    G.down.P.uin = S.u.p;
    G.down.P.e = nullptr;
    G.down.P.uout = S.tmp.p;
    G.down.P.fc = lv[l + 1].f.p;
    fill(G.up);
    G.up.P.uin = S.tmp.p;
    G.up.P.e = lv[l + 1].u.p;
    G.up.P.uout = S.u.p;
    G.up.P.fc = nullptr;
    leg_dispatch(G.down, 0, nullptr);
    leg_dispatch(G.up, 0, nullptr);
    G.ok = true;
  }
  bool leg_ok(int l) const { return l >= 0 && l < (int)legs.size() && legs[l].ok; }
  std::vector<char> leg_side;  // per level: this cycle's down-leg result exchange went to the side stream

  // ---- coarse tail (k_coarse_tail): levels [tail_first, L) of a damped-Jacobi cycle in one launch
  int tail_first = -1;
  dev::TailParams tail{};
  size_t tail_smem = 0;
  void prepare_tail() {
    tail_first = -1;
    if (!(opt.fuse & 16) || opt.smoother != AMGB_SMOOTHER_JACOBI || opt.smoother_iters < 1 || L < 2 ||
        !opt.skip_dead_coarse_smooth)
      return;
    const int bw = factor.bw, nc = factor.n;
    const size_t smem = sizeof(double) * (size_t)nc * (std::max(bw, 1) + 1);
    if (bw < 1 || bw > 8 || smem > 200 * 1024) return;
    const int64_t max_rows = env_int("AMGB_TAIL_ROWS", (opt.fuse & 32) ? 1100 : 6000);  // with the mid kernels on, only the smallest levels
    int first = L - 1;  // the coarsest level alone is just the solve
    while (first - 1 >= 1 && first - 1 >= L - 1 - dev::kTailMaxLevels && n[first - 1] <= max_rows) {
      const int l = first - 1;
      const LevelState& S = lv[l];
      const DevMat& A = ops[l]->rows_of_A();
      bool has_diag = false;
      if (A.is_dia)
        for (int d = 0; d < A.dia.n_diag; ++d) has_diag |= (A.dia.off[d] == 0);
      if (S.sharded || !S.tmp.p || !A.is_dia || A.dia.n_diag > 10 || A.dia.rows.p || !has_diag) break;
      first = l;
    }
    if (first >= L - 1) return;  // nothing to fuse
    tail = dev::TailParams{};
    tail.n_tail = L - 1 - first;
    tail.nu = (int)opt.smoother_iters;
    tail.omega = opt.omega;
    tail.nc = nc;
    tail.bw = bw;
    tail.L = dL.p;
    tail.d = dd.p;
    tail.f_c = lv[L - 1].f.p;
    tail.u_c = lv[L - 1].u.p;
    for (int l = first; l < L - 1; ++l) {
      dev::TailLevel& V = tail.lv[l - first];
      const DevMat& A = ops[l]->rows_of_A();
      V.A = A.dia.view();
      V.A.mask = nullptr;  // every diagonal is read (the per-slice masks do not pay on tiny levels)
      V.A.n_rows = (int)n[l];
      V.diag_d = 0;
      for (int d = 0; d < A.dia.n_diag; ++d)
        if (A.dia.off[d] == 0) V.diag_d = d;
      V.n = (int)n[l];
      V.n_coarse = (int)n[l + 1];
      V.f = lv[l].f.p;
      V.u = lv[l].u.p;
      V.tmp = lv[l].tmp.p;
      V.f_coarse = lv[l + 1].f.p;
    }
    tail_smem = smem;
    if (smem > 48 * 1024)
      CUDA_CHECK(cudaFuncSetAttribute(dev::k_coarse_tail, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    tail_first = first;
  }
  void launch_tail(cudaStream_t s) { LAUNCH(dev::k_coarse_tail, 1, 1024, tail_smem, s, tail); }

  // ---- mid levels (mid_levels.cuh): levels [mid_first, mid_end) of a damped-Jacobi cycle, all their
  // down legs in ONE launch and all their up legs in another (option fuse bit 5)
  int mid_first = -1, mid_end = -1;
  mid::Params midp{};
  void prepare_mid() {
    mid_first = mid_end = -1;
    if (!(opt.fuse & 32) || opt.smoother != AMGB_SMOOTHER_JACOBI || opt.smoother_iters < 1 || L < 2 ||
        !opt.skip_dead_coarse_smooth)
      return;
    const int end = (tail_first > 0) ? tail_first : L - 1;  // the level below the last mid level
    const int64_t max_rows = env_int("AMGB_MID_ROWS", 70000);
    auto eligible = [&](int l) {
      if (l < 0 || l >= end) return false;
      const LevelState& S = lv[l];
      const DevMat& A = ops[l]->rows_of_A();
      if (S.sharded || !S.tmp.p || !A.is_dia || A.dia.n_diag > mid::kMaxDiag || A.dia.rows.p || n[l] > max_rows) return false;
      bool has_diag = false;
      for (int d = 0; d < A.dia.n_diag; ++d) has_diag |= (A.dia.off[d] == 0);
      return has_diag;
    };
    int first = end;
    while (first - 1 >= 0 && end - (first - 1) <= mid::kMaxLevels && eligible(first - 1)) --first;
    for (; first < end; ++first) {  // drop the finest candidate until a tile layout fits shared memory
      mid::Params P{};
      P.n_lv = end - first;
      P.nu = (int)opt.smoother_iters;
      P.first_is_level0 = (first == 0);
      P.omega = opt.omega;
      for (int l = first; l < end; ++l) {
        mid::Level& V = P.lv[l - first];
        const DevDia& D = ops[l]->rows_of_A().dia;
        V.n = (int)n[l];
        V.n_coarse = (int)n[l + 1];
        V.nd = D.n_diag;
        V.w = 0;
        for (int d = 0; d < D.n_diag; ++d) {
          V.off[d] = D.off[d];
          if (D.off[d] == 0) V.diag_d = d;
          V.w = std::max(V.w, std::abs(D.off[d]));
        }
        V.ld = D.ld;
        V.val = D.val.p;
        V.f = lv[l].f.p;
        V.u = lv[l].u.p;
        V.tmp = lv[l].tmp.p;
      }
      P.f_next = lv[end].f.p;
      P.u_next = lv[end].u.p;
      P.n_next = (int)n[end];
      if (mid::plan_layout(P, 200 * 1024 / 8)) {
        midp = P;
        mid_first = first;
        mid_end = end;
        const int bytes = 8 * std::max(P.smem_doubles_down, P.smem_doubles_up);
        if (bytes > 48 * 1024) {
          CUDA_CHECK(cudaFuncSetAttribute(mid::k_mid<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
          CUDA_CHECK(cudaFuncSetAttribute(mid::k_mid<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
          CUDA_CHECK(cudaFuncSetAttribute(mid::k_mid<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
          CUDA_CHECK(cudaFuncSetAttribute(mid::k_mid<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
        }
        return;
      }
    }
  }
  void mid_down(cudaStream_t s) {
    const size_t bytes = 8 * (size_t)midp.smem_doubles_down;
    const int threads = env_int("AMGB_MID_THREADS", 1024);
    if (fast_arith()) LAUNCH((mid::k_mid<true, false>), midp.n_blocks, threads, bytes, s, midp);
    else LAUNCH((mid::k_mid<false, false>), midp.n_blocks, threads, bytes, s, midp);
  }
  void mid_up(cudaStream_t s) {
    const size_t bytes = 8 * (size_t)midp.smem_doubles_up;
    const int threads = env_int("AMGB_MID_THREADS", 1024);
    if (fast_arith()) LAUNCH((mid::k_mid<true, true>), midp.n_blocks, threads, bytes, s, midp);
    else LAUNCH((mid::k_mid<false, true>), midp.n_blocks, threads, bytes, s, midp);
  }

  // optional phase marks (amgb_hierarchy_phase_times): events recorded at the phase boundaries of an
  // un-captured cycle -- [0] start, [1] sharded down legs done, [2] gather done, [3] replicated /
  // single-GPU coarse part done (levels below the sharded ones, both directions), [4] end
  cudaEvent_t* phase_ev = nullptr;
  void mark(int i, cudaStream_t s) {
    if (phase_ev) CUDA_CHECK(cudaEventRecord(phase_ev[i], s));
  }
  void enqueue_vcycle(cudaStream_t s) {
    halo_exchanges_per_vcycle = 0;
    site_cursor = 0;  // sites 0 .. k-1 belong to the V-cycle, in the same order on every rank
    const int lt = (tail_first > 0) ? tail_first : L;  // levels [lt, L) run inside k_coarse_tail
    const int lm = (mid_first >= 0) ? mid_first : lt;  // levels [lm, mid_end) run inside the mid kernels
    mark(0, s);
    if (n_sharded == 0) {
      mark(1, s);
      mark(2, s);
    }
    for (int l = 0; l < lm; ++l) {
      const bool coarsest = (l + 1 == L);
      if (coarsest && opt.skip_dead_coarse_smooth) break;
      if (leg_ok(l)) {  // sweeps + residual + restriction in one pass: u_l -> tmp_l, f_{l+1}
        if (lv[l].sharded && fused_push) {
          // the leg waits for the neighbours' previous site itself and pushes its boundary rows
          leg_down(l, s);
          if (!lv[l + 1].sharded) {  // first agglomerated level: every rank gets the whole right-hand side
            mark(1, s);
            gather_coarse_rhs(s);
            mark(2, s);
          }
        } else if (lv[l].sharded) {
          // ghost rows of the leg's input: the iterate on level 0, the right-hand side below
          exchange(l, l == 0 ? lv[l].u.p : lv[l].fw.p, s);
          leg_down(l, s);
          // The up leg needs the ghost rows of this result: exchange them now on the side stream,
          // while the coarser levels run, instead of on the way back up.
          leg_side[l] = p2p && overlap && aux_stream && l < (int)ev_leg.size();  // (NCCL calls stay on one stream)
          if (leg_side[l]) {
            CUDA_CHECK(cudaEventRecord(ev_fork, s));
            CUDA_CHECK(cudaStreamWaitEvent(aux_stream, ev_fork, 0));
            exchange(l, lv[l].tmp.p, aux_stream);
            CUDA_CHECK(cudaEventRecord(ev_leg[l], aux_stream));
          }
          if (!lv[l + 1].sharded) {  // first agglomerated level: every rank gets the whole right-hand side
            mark(1, s);
            gather_coarse_rhs(s);
            mark(2, s);
          }
        } else {
          leg_down(l, s);
        }
        continue;
      }
      // a fused finer level does not zero u_l (its own coarse levels never read it)
      if (l > 0 && leg_ok(l - 1)) CUDA_CHECK(cudaMemsetAsync(lv[l].u.p, 0, sizeof(double) * lv[l].u.n, s));
      smooth(l, s, /*from_zero=*/l > 0);
      const bool last_sharded = lv[l].sharded && !coarsest && !lv[l + 1].sharded;
      if (last_sharded) mark(1, s);  // (per-operator sharded path: the gather happens inside residual_restrict)
      if (!coarsest) residual_restrict(l, s);
      if (last_sharded) mark(2, s);
      // on the coarsest level the reference also forms the residual (:272-274);
      // it is stored in a private member without a getter and never read.
    }
    if (mid_first >= 0) mid_down(s);
    if (lt < L) launch_tail(s);
    else coarse_solve(s);
    if (mid_first >= 0) mid_up(s);
    if (n_sharded == 0) mark(3, s);
    for (int l = std::min(lm, L - 1) - 1; l >= 0; --l) {
      if (l == n_sharded - 1) mark(3, s);
      if (leg_ok(l)) {  // tmp_l + P u_{l+1}, sweeps -> u_l
        if (lv[l].sharded && !fused_push) {
          if (leg_side[l]) CUDA_CHECK(cudaStreamWaitEvent(s, ev_leg[l], 0));
          else exchange(l, lv[l].tmp.p, s);
          if (lv[l + 1].sharded) exchange(l + 1, lv[l + 1].u.p, s);
        }
        leg_up(l, s);
      } else {
        smooth(l, s, false, /*with_prolong=*/true);
      }
    }
    mark(4, s);
  }
  void build_graph() {
    if (exec) return;
    const int64_t before = g_launches.load();
    CUDA_CHECK(cudaStreamBeginCapture(own_stream, cudaStreamCaptureModeThreadLocal));
    try {
      enqueue_vcycle(own_stream);
    } catch (...) {
      cudaGraph_t g = nullptr;
      cudaStreamEndCapture(own_stream, &g);
      if (g) cudaGraphDestroy(g);
      throw;
    }
    CUDA_CHECK(cudaStreamEndCapture(own_stream, &graph));
    CUDA_CHECK(cudaGraphInstantiate(&exec, graph, 0));
    launches_per_vcycle = g_launches.load() - before;
    g_launches.store(before);  // capture itself launched nothing
  }
  void vcycle() {
    if (opt.use_graph) {
      build_graph();
      CUDA_CHECK(cudaGraphLaunch(exec, stream));
      g_launches.fetch_add(launches_per_vcycle, std::memory_order_relaxed);
    } else {
      const int64_t before = g_launches.load();
      enqueue_vcycle(stream);
      launches_per_vcycle = g_launches.load() - before;
    }
  }
  // sum over all ranks of a device scalar, returned on the host
  double finish_scalar() {
    if (comm && world() > 1)
      NCCL_CHECK(NcclApi::get().AllReduce(scalar.p, scalar.p, 1, ncclDouble, ncclSum, comm->comm, stream));
    double out = 0.0;
    CUDA_CHECK(cudaMemcpyAsync(&out, scalar.p, sizeof(double), cudaMemcpyDeviceToHost, stream));
    CUDA_CHECK(cudaStreamSynchronize(stream));
    check_halo();
    return out;
  }
  double rss() {
    LevelState& S = lv[0];
    if (S.sharded) exchange_outside_cycle(0, S.u.p);
    ops[0]->rss(S.u_own(), S.f.p, partial.p, scalar.p, stream);
    return S.sharded ? finish_scalar() : finish_scalar_local();
  }
  double finish_scalar_local() {
    double out = 0.0;
    CUDA_CHECK(cudaMemcpyAsync(&out, scalar.p, sizeof(double), cudaMemcpyDeviceToHost, stream));
    CUDA_CHECK(cudaStreamSynchronize(stream));
    return out;
  }
  // sum of squares of the level-0 rhs
  double rhs_sumsq() {
    LevelState& S = lv[0];
    const int nb = std::max(1, blocks_for(S.n_own, 256));
    LAUNCH(dev::k_sumsq_partial, nb, 256, 0, stream, S.f.p, S.n_own, partial.p);
    LAUNCH(dev::k_sum_partials, 1, 256, 0, stream, partial.p, nb, scalar.p);
    return S.sharded ? finish_scalar() : finish_scalar_local();
  }
  void check_level(int l, bool need_next = false) const {
    if (l < 0 || l >= L || (need_next && l + 1 >= L)) throw std::invalid_argument("level out of range");
  }
  void require_whole(int l) const {
    if (lv[l].sharded)
      throw ApiError(AMGB_ESTATE, "this per-operator entry point is not available on a sharded level");
  }

  // ---- host <-> device copies of a level vector given / returned at full length ----
  void upload_u(int l, const double* full) {
    LevelState& S = lv[l];
    if (!S.sharded) {
      CUDA_CHECK(cudaMemcpyAsync(S.u.p, full, sizeof(double) * n[l], cudaMemcpyHostToDevice, stream));
    } else {
      const int64_t lo = std::max<int64_t>(0, S.s - S.halo_lo), hi = std::min<int64_t>(n[l], S.e + S.halo_hi);
      CUDA_CHECK(cudaMemcpyAsync(S.u.p + (lo - (S.s - S.halo_lo)), full + lo, sizeof(double) * (hi - lo),
                                 cudaMemcpyHostToDevice, stream));
    }
    CUDA_CHECK(cudaStreamSynchronize(stream));
  }
  void upload_f(int l, const double* full) {
    LevelState& S = lv[l];
    if (S.sharded && S.fw.p) {
      const int64_t lo = std::max<int64_t>(0, S.s - S.halo_lo), hi = std::min<int64_t>(n[l], S.e + S.halo_hi);
      CUDA_CHECK(cudaMemcpyAsync(S.fw.p + (lo - (S.s - S.halo_lo)), full + lo, sizeof(double) * (hi - lo),
                                 cudaMemcpyHostToDevice, stream));
    }
    CUDA_CHECK(cudaMemcpyAsync(S.f.p, full + S.s, sizeof(double) * S.n_mat, cudaMemcpyHostToDevice, stream));
    CUDA_CHECK(cudaStreamSynchronize(stream));
  }
  // ---- device-side setup (setup_dia.cuh): the level-0 CSC as handed in stays on the device; the host
  // copies of the level matrices (structural CSC, explicit zeros kept) that the getters return are
  // rebuilt on demand with the host Galerkin chain
  bool device_setup = false;
  int raw_rows = 0;
  DevBuf<int> raw_colptr, raw_rowidx;
  DevBuf<double> raw_val;
  std::vector<Csc> host_mats;
  const Csc& host_matrix(int level) {
    if (sa_resident) {
      if (host_mats.empty()) host_mats.resize(L);
      if (host_mats[level].colptr.empty()) host_mats[level] = sa_dev_A[level].download(stream);
      return host_mats[level];
    }
    if (!device_setup || sa()) return ops[level]->M;
    if (host_mats.empty()) {
      host_mats.resize(1);
      Csc& A = host_mats[0];
      A.rows = A.cols = raw_rows;
      A.colptr.resize(raw_colptr.n);
      A.rowidx.resize(raw_rowidx.n);
      A.val.resize(raw_val.n);
      CUDA_CHECK(cudaMemcpy(A.colptr.data(), raw_colptr.p, raw_colptr.n * sizeof(int), cudaMemcpyDeviceToHost));
      CUDA_CHECK(cudaMemcpy(A.rowidx.data(), raw_rowidx.p, raw_rowidx.n * sizeof(int), cudaMemcpyDeviceToHost));
      CUDA_CHECK(cudaMemcpy(A.val.data(), raw_val.p, raw_val.n * sizeof(double), cudaMemcpyDeviceToHost));
    }
    while ((int)host_mats.size() <= level) {  // multigrid.hpp:211-223
      const int l = (int)host_mats.size();
      Csc P = prolongation(l - 1);
      Csc R = transpose(P);
      host_mats.push_back(galerkin(R, host_mats[l - 1], P));
    }
    return host_mats[level];
  }

  DevBuf<double> gather_buf;  // full-length staging vector of the sharded getters (allocated on first use)
  void download(int l, bool want_u, double* full) {
    LevelState& S = lv[l];
    if (!S.sharded) {
      CUDA_CHECK(cudaMemcpyAsync(full, want_u ? S.u.p : S.f.p, sizeof(double) * n[l],
                                 cudaMemcpyDeviceToHost, stream));
    } else {
      // every rank returns the whole vector: gather the blocks over NVLink into a persistent
      // staging vector, then one D2H copy.  (Callers that own a row block use download_local.)
      if (gather_buf.n < (size_t)n[l]) gather_buf.alloc(n[l]);
      CUDA_CHECK(cudaMemcpyAsync(gather_buf.p + S.s, want_u ? S.u_own() : S.f.p, sizeof(double) * S.n_own,
                                 cudaMemcpyDeviceToDevice, stream));
      allgather_blocks(gather_buf.p, plan.start[l], stream);
      CUDA_CHECK(cudaMemcpyAsync(full, gather_buf.p, sizeof(double) * n[l], cudaMemcpyDeviceToHost, stream));
    }
    CUDA_CHECK(cudaStreamSynchronize(stream));
    check_halo();
  }
  // this rank's rows [s, e) only: no collective, 1/world of the bytes
  void download_local(int l, bool want_u, double* block) {
    LevelState& S = lv[l];
    CUDA_CHECK(cudaMemcpyAsync(block, want_u ? S.u_own() : S.f.p, sizeof(double) * S.n_own,
                               cudaMemcpyDeviceToHost, stream));
    CUDA_CHECK(cudaStreamSynchronize(stream));
    check_halo();
  }
  // out-of-cycle halo exchange of a level vector (reserved site; collective over the ranks)
  void exchange_outside_cycle(int l, double* base) {
    const int keep = site_cursor;
    site_cursor = kMaxSites - 1;
    exchange(l, base, stream);
    site_cursor = keep;
  }
  void upload_local(int l, bool want_u, const double* block) {
    LevelState& S = lv[l];
    if (want_u) {
      CUDA_CHECK(cudaMemcpyAsync(S.u_own(), block, sizeof(double) * S.n_own, cudaMemcpyHostToDevice, stream));
      if (S.sharded) exchange_outside_cycle(l, S.u.p);
    } else {
      CUDA_CHECK(cudaMemcpyAsync(S.f.p, block, sizeof(double) * S.n_own, cudaMemcpyHostToDevice, stream));
      if (S.sharded) {
        if (S.fw.p) {
          CUDA_CHECK(cudaMemcpyAsync(S.fw.p + S.halo_lo, S.f.p, sizeof(double) * S.n_own, cudaMemcpyDeviceToDevice,
                                     stream));
          exchange_outside_cycle(l, S.fw.p);
          // the per-operator kernels read f on the ghost rows [n_own, n_mat) too
          if (S.n_mat > S.n_own)
            CUDA_CHECK(cudaMemcpyAsync(S.f.p + S.n_own, S.fw.p + S.halo_lo + S.n_own,
                                       sizeof(double) * (S.n_mat - S.n_own), cudaMemcpyDeviceToDevice, stream));
        } else if (S.n_mat > S.n_own) {
          throw ApiError(AMGB_ESTATE, "set_rhs_local needs the window layout on this level");
        }
      }
    }
    CUDA_CHECK(cudaStreamSynchronize(stream));
    check_halo();
  }
};

// ============================================================================
// C ABI
// ============================================================================
extern "C" {

const char* amgb_last_error(void) { return g_err.c_str(); }
int amgb_version(void) { return 100; }
int amgb_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}
int amgb_set_device(int device) {
  return guarded([&] { CUDA_CHECK(cudaSetDevice(device)); });
}

// ---- generators / setup helpers (host only) ----
double amgb_grid_spacing_h(int64_t n) { return grid_spacing_h(n); }
int64_t amgb_points_n_from_grid_spacing_h(double h) { return (int64_t)((2 / h) - 1); }  // grid.hpp:39-41
int64_t amgb_grid_laplacian_nnz(int64_t n) { return 5 * n * n - 4 * n; }
int amgb_grid_laplacian(int64_t n, double eps_y, int* colptr, int* rowidx, double* val) {
  return guarded([&] {
    if (n < 1 || n * n > 2147483647LL / 5) throw std::invalid_argument("grid size out of range");
    Csc A = grid_laplacian(n, eps_y);
    std::memcpy(colptr, A.colptr.data(), A.colptr.size() * sizeof(int));
    std::memcpy(rowidx, A.rowidx.data(), A.rowidx.size() * sizeof(int));
    std::memcpy(val, A.val.data(), A.val.size() * sizeof(double));
  });
}
int amgb_grid_rhs(int64_t n, double* b) {
  return guarded([&] {
    if (n < 1) throw std::invalid_argument("grid size out of range");
    grid_rhs(n, b);
  });
}
int64_t amgb_n_H_dofs_from_n_h_dofs(int64_t n_h) { return coarse_dofs(n_h); }
int64_t amgb_interp_nnz(int64_t n_h, int64_t n_H) {
  int64_t c = 0;
  for (int64_t j = 0; j < n_H; ++j) c += (2 * j < n_h) + (2 * j + 1 < n_h) + (2 * j + 2 < n_h);
  return c;
}
int amgb_interp_make_operators(int64_t n_h, int64_t n_H, int* P_colptr, int* P_rowidx, double* P_val,
                               int* R_colptr, int* R_rowidx, double* R_val) {
  return guarded([&] {
    if (n_h < 0 || n_H < 0) throw std::invalid_argument("negative size");
    Csc P = make_prolongation(n_h, n_H);
    Csc R = transpose(P);
    std::memcpy(P_colptr, P.colptr.data(), P.colptr.size() * sizeof(int));
    std::memcpy(P_rowidx, P.rowidx.data(), P.rowidx.size() * sizeof(int));
    std::memcpy(P_val, P.val.data(), P.val.size() * sizeof(double));
    std::memcpy(R_colptr, R.colptr.data(), R.colptr.size() * sizeof(int));
    std::memcpy(R_rowidx, R.rowidx.data(), R.rowidx.size() * sizeof(int));
    std::memcpy(R_val, R.val.data(), R.val.size() * sizeof(double));
  });
}

int64_t amgb_bilinear_coarse_lines(int64_t m_h) { return m_h < 0 ? -1 : coarse_lines_2d(m_h); }
int64_t amgb_bilinear_nnz(int64_t m_h, int64_t m_H) {
  const int64_t k = amgb_interp_nnz(m_h, m_H);
  return k < 0 ? -1 : k * k;
}
int amgb_bilinear_make_operators(int64_t m_h, int64_t m_H, int* P_colptr, int* P_rowidx, double* P_val,
                                 int* R_colptr, int* R_rowidx, double* R_val) {
  return guarded([&] {
    if (m_h < 0 || m_H < 0) throw std::invalid_argument("negative size");
    if (!P_colptr || !P_rowidx || !P_val || !R_colptr || !R_rowidx || !R_val) throw std::invalid_argument("null argument");
    const Csc P = make_prolongation_2d(m_h, m_H);
    const Csc R = transpose(P);
    std::memcpy(P_colptr, P.colptr.data(), P.colptr.size() * sizeof(int));
    std::memcpy(P_rowidx, P.rowidx.data(), P.rowidx.size() * sizeof(int));
    std::memcpy(P_val, P.val.data(), P.val.size() * sizeof(double));
    std::memcpy(R_colptr, R.colptr.data(), R.colptr.size() * sizeof(int));
    std::memcpy(R_rowidx, R.rowidx.data(), R.rowidx.size() * sizeof(int));
    std::memcpy(R_val, R.val.data(), R.val.size() * sizeof(double));
  });
}
int amgb_sa_aggregate(int n, const int* colptr, const int* rowidx, const double* val, double theta, int* agg,
                      int64_t* n_aggregates) {
  return guarded([&] {
    if (n < 0 || !colptr || !rowidx || !val || !agg || !n_aggregates) throw std::invalid_argument("null argument");
    std::vector<int> a;
    *n_aggregates = sa_aggregate(csc_from_arrays(n, n, colptr, rowidx, val), theta, a);
    std::memcpy(agg, a.data(), a.size() * sizeof(int));
  });
}
int amgb_linear_restrict(int64_t n_h, int64_t n_H, const double* r, double* out) {
  return guarded([&] {
    if (!r || !out || n_h < 0 || n_H < 0) throw std::invalid_argument("bad transfer arguments");
    require_device();
    DevBuf<double> dr, dout;
    dr.upload(r, n_h, nullptr);
    dout.alloc(n_H);
    if (n_H) LAUNCH(dev::k_restrict, blocks_for(n_H, 256), 256, 0, nullptr, dr.p, (int)n_h, dout.p, (int)n_H);
    dout.download(out, nullptr);
    CUDA_CHECK(cudaStreamSynchronize(nullptr));
  });
}
int amgb_linear_prolong(int64_t n_h, int64_t n_H, const double* e, double* out) {
  return guarded([&] {
    if (!e || !out || n_h < 0 || n_H < 0) throw std::invalid_argument("bad transfer arguments");
    require_device();
    DevBuf<double> de, dout;
    de.upload(e, n_H, nullptr);
    dout.alloc(n_h);
    dout.zero(nullptr);
    if (n_h)
      LAUNCH(dev::k_prolong_add, blocks_for(n_h, 256), 256, 0, nullptr, de.p, 0, (int)n_H, dout.p, 0, (int)n_h);
    dout.download(out, nullptr);
    CUDA_CHECK(cudaStreamSynchronize(nullptr));
  });
}

// y = A x for any CSC matrix (rectangular too), Eigen's evaluation order: the stored P / R of an
// InterpolatorBase applied as get_P(level) * v (interpolator.hpp:52-68).  One-shot: the matrix
// is mirrored (rows of A, SELL-32 or DIA), applied and dropped.
int amgb_csc_spmv(int n_rows, int n_cols, const int* colptr, const int* rowidx, const double* val,
                  const double* x, double* y) {
  return guarded([&] {
    if (!colptr || !x || !y || n_rows < 0 || n_cols < 0) throw std::invalid_argument("bad spmv arguments");
    require_device();
    Csc AT = transpose(csc_from_arrays(n_rows, n_cols, colptr, rowidx, val));  // column k of AT = row k of A
    DevMat M;
    M.upload(AT, nullptr, nullptr);
    DevBuf<double> dx, dy;
    dx.upload(x, n_cols, nullptr);
    dy.alloc(n_rows);
    if (n_rows)
      with_view(M, [&](auto V) {
        auto kern = dev::k_spmv<decltype(V)>;
        V.n_rows = n_rows;
        LAUNCH(kern, blocks_for(n_rows, 256), 256, 0, nullptr, V, dx.p, dy.p);
      });
    dy.download(y, nullptr);
    CUDA_CHECK(cudaStreamSynchronize(nullptr));
  });
}

// ---- amgb_matrix ----
int amgb_matrix_create(int n_rows, int n_cols, const int* colptr, const int* rowidx, const double* val,
                       amgb_matrix** out) {
  return guarded([&] {
    if (!out || !colptr || n_rows < 0 || n_cols < 0) throw std::invalid_argument("bad matrix arguments");
    require_device();
    std::unique_ptr<amgb_matrix> m(new amgb_matrix());
    CUDA_CHECK(cudaGetDevice(&m->device));
    CUDA_CHECK(cudaStreamCreateWithFlags(&m->stream, cudaStreamNonBlocking));
    m->op.build(csc_from_arrays(n_rows, n_cols, colptr, rowidx, val), m->stream);
    m->u.alloc(n_cols);
    m->b.alloc(n_cols);
    m->r.alloc((size_t)n_cols + 4);
    m->partial.alloc(m->op.rss_blocks());
    m->scalar.alloc(1);
    *out = m.release();
  });
}
int amgb_matrix_destroy(amgb_matrix* A) {
  return guarded([&] {
    if (!A) return;
    cudaSetDevice(A->device);
    delete A;
  });
}
int64_t amgb_matrix_nnz_device(const amgb_matrix* A) { return A ? A->op.nnz_device() : 0; }
int amgb_matrix_is_symmetric(const amgb_matrix* A) { return A && A->op.symmetric; }

static double matrix_rss(amgb_matrix* A) {
  A->op.rss(A->u.p, A->b.p, A->partial.p, A->scalar.p, A->stream);
  double out = 0.0;
  CUDA_CHECK(cudaMemcpyAsync(&out, A->scalar.p, sizeof(double), cudaMemcpyDeviceToHost, A->stream));
  CUDA_CHECK(cudaStreamSynchronize(A->stream));
  return out;
}

int amgb_smooth_gs(amgb_matrix* A, double* u, const double* b, double tolerance, int64_t every,
                   int64_t n_iters, int mode, int64_t* iters_done, double* final_error) {
  return guarded([&] {
    if (!A || !u || !b) throw std::invalid_argument("null argument");
    CUDA_CHECK(cudaSetDevice(A->device));
    cudaStream_t s = A->stream;
    A->u.upload(u, A->op.n, s);
    A->b.upload(b, A->op.n, s);
    int64_t iter = 0;
    double error = 100;
    while (iter < n_iters && error > tolerance) {  // smoother.hpp:195-203
      A->op.gs_direction(true, A->b.p, A->u.p, A->r.p, mode, s);
      A->op.gs_direction(false, A->b.p, A->u.p, A->r.p, mode, s);
      iter += 1;
      if (every != 0 && iter % every == 0) error = matrix_rss(A);
    }
    A->u.download(u, s);
    CUDA_CHECK(cudaStreamSynchronize(s));
    if (iters_done) *iters_done = iter;
    if (final_error) *final_error = error;
  });
}
int amgb_smooth_jacobi(amgb_matrix* A, double* u, const double* b, double omega, int64_t n_sweeps) {
  return guarded([&] {
    if (!A || !u || !b) throw std::invalid_argument("null argument");
    CUDA_CHECK(cudaSetDevice(A->device));
    cudaStream_t s = A->stream;
    A->u.upload(u, A->op.n, s);
    A->b.upload(b, A->op.n, s);
    double* src = A->u.p;
    double* dst = A->r.p;
    for (int64_t it = 0; it < n_sweeps; ++it) {
      A->op.jacobi(src, A->b.p, omega, dst, s);
      std::swap(src, dst);
    }
    if (A->op.n) CUDA_CHECK(cudaMemcpyAsync(u, src, sizeof(double) * A->op.n, cudaMemcpyDeviceToHost, s));
    CUDA_CHECK(cudaStreamSynchronize(s));
  });
}
int amgb_smooth_color_gs(amgb_matrix* A, double* u, const double* b, int64_t n_iters) {
  return guarded([&] {
    if (!A || !u || !b) throw std::invalid_argument("null argument");
    CUDA_CHECK(cudaSetDevice(A->device));
    cudaStream_t s = A->stream;
    A->op.ensure_colors(s);
    A->u.upload(u, A->op.n, s);
    A->b.upload(b, A->op.n, s);
    for (int64_t it = 0; it < n_iters; ++it) {
      for (int c = 0; c < A->op.n_colors; ++c) A->op.color_pass(c, A->b.p, A->u.p, s);
      for (int c = A->op.n_colors - 1; c >= 0; --c) A->op.color_pass(c, A->b.p, A->u.p, s);
    }
    A->u.download(u, s);
    CUDA_CHECK(cudaStreamSynchronize(s));
  });
}
int amgb_smooth_line_gs(amgb_matrix* A, double* u, const double* b, int64_t n_iters, int lines) {
  return guarded([&] {
    if (!A || !u || !b) throw std::invalid_argument("null argument");
    if (lines != AMGB_LINES_X && lines != AMGB_LINES_Y && lines != AMGB_LINES_ALTERNATING)
      throw std::invalid_argument("unknown line direction setting " + std::to_string(lines));
    const int m = (int)grid_lines(A->op.n);
    if (m < 1) throw std::invalid_argument("line Gauss-Seidel needs an m x m grid operator (rows not a square number)");
    CUDA_CHECK(cudaSetDevice(A->device));
    cudaStream_t s = A->stream;
    A->op.ensure_line_gs_lines(m, lines, false, "the matrix", s);
    A->u.upload(u, A->op.n, s);
    A->b.upload(b, A->op.n, s);
    for (int64_t it = 0; it < n_iters; ++it) {
      A->op.line_gs_half(true, lines, false, A->b.p, A->u.p, A->r.p, s);
      A->op.line_gs_half(false, lines, false, A->b.p, A->u.p, A->r.p, s);
    }
    A->u.download(u, s);
    CUDA_CHECK(cudaStreamSynchronize(s));
  });
}
int amgb_matrix_coloring(amgb_matrix* A, int* n_colors, int* color) {
  return guarded([&] {
    if (!A) throw std::invalid_argument("null argument");
    CUDA_CHECK(cudaSetDevice(A->device));
    A->op.ensure_colors(A->stream);
    if (n_colors) *n_colors = A->op.n_colors;
    if (color) std::memcpy(color, A->op.color.data(), sizeof(int) * A->op.color.size());
  });
}
int amgb_residual(amgb_matrix* A, const double* u, const double* f, double* r) {
  return guarded([&] {
    if (!A || !u || !f || !r) throw std::invalid_argument("null argument");
    CUDA_CHECK(cudaSetDevice(A->device));
    cudaStream_t s = A->stream;
    A->u.upload(u, A->op.n, s);
    A->b.upload(f, A->op.n, s);
    A->op.residual(A->u.p, A->b.p, A->r.p, s);
    if (A->op.n) CUDA_CHECK(cudaMemcpyAsync(r, A->r.p, sizeof(double) * A->op.n, cudaMemcpyDeviceToHost, s));
    CUDA_CHECK(cudaStreamSynchronize(s));
  });
}
int amgb_rss(amgb_matrix* A, const double* u, const double* b, double* out) {
  return guarded([&] {
    if (!A || !u || !b || !out) throw std::invalid_argument("null argument");
    CUDA_CHECK(cudaSetDevice(A->device));
    A->u.upload(u, A->op.n, A->stream);
    A->b.upload(b, A->op.n, A->stream);
    *out = matrix_rss(A);
  });
}

// Mean milliseconds per launch of one pass over the matrix on the vectors of the last call that
// uploaded them (amgb_residual / amgb_rss): kind 0 one damped-Jacobi sweep, 1 one colour-complete
// multicolour Gauss-Seidel sweep (every colour once), 2 one residual.  CUDA events on the handle's stream.
int amgb_matrix_time(amgb_matrix* A, int kind, double omega, int warmup, int reps, double* ms_out) {
  return guarded([&] {
    if (!A || !ms_out || reps < 1 || kind < 0 || kind > 4) throw std::invalid_argument("bad argument");
    CUDA_CHECK(cudaSetDevice(A->device));
    cudaStream_t s = A->stream;
    if (A->u.n != (size_t)A->op.n || A->b.n != (size_t)A->op.n)
      throw ApiError(AMGB_ESTATE, "upload vectors first (amgb_residual / amgb_rss)");
    if (kind == 1) A->op.ensure_colors(s);
    double* src = A->u.p;
    double* dst = A->r.p;
    auto once = [&] {
      if (kind == 0) {
        A->op.jacobi(src, A->b.p, omega, dst, s);
        std::swap(src, dst);
      } else if (kind == 1) {
        for (int c = 0; c < A->op.n_colors; ++c) A->op.color_pass(c, A->b.p, A->u.p, s);
      } else if (kind >= 3) {
        A->op.gs_direction(true, A->b.p, A->u.p, A->r.p, kind == 3 ? AMGB_GS_AUTO : AMGB_GS_LINESCAN, s);
      } else {
        A->op.residual(A->u.p, A->b.p, A->r.p, s);
      }
    };
    for (int i = 0; i < warmup; ++i) once();
    cudaEvent_t e0, e1;
    CUDA_CHECK(cudaEventCreate(&e0));
    CUDA_CHECK(cudaEventCreate(&e1));
    CUDA_CHECK(cudaEventRecord(e0, s));
    for (int i = 0; i < reps; ++i) once();
    CUDA_CHECK(cudaEventRecord(e1, s));
    CUDA_CHECK(cudaEventSynchronize(e1));
    float ms = 0.f;
    CUDA_CHECK(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    *ms_out = (double)ms / reps;
  });
}
int amgb_selftest_division(int64_t n_pairs, uint64_t seed, int64_t* mismatches) {
  return guarded([&] {
    if (!mismatches || n_pairs < 0) throw std::invalid_argument("bad argument");
    DevBuf<unsigned long long> count;
    count.alloc(1);
    count.zero(nullptr);
    LAUNCH(gsw::k_gsw_division_selftest, 1184, 256, 0, nullptr, (long long)n_pairs, (unsigned long long)seed, count.p);
    unsigned long long got = 0;
    CUDA_CHECK(cudaMemcpy(&got, count.p, sizeof(got), cudaMemcpyDeviceToHost));
    *mismatches = (int64_t)got;
  });
}
int amgb_matrix_gs_kernel(amgb_matrix* A, int mode) {
  int kind = -1;
  const int rc = guarded([&] {
    if (!A) throw std::invalid_argument("null argument");
    CUDA_CHECK(cudaSetDevice(A->device));
    kind = A->op.gs_kernel(mode, A->stream);
  });
  return rc == AMGB_OK ? kind : -1;
}
// bytes of matrix data one pass streams: kind 0 / 2 the rows-of-A mirror, kind 1 the per-colour mirrors
int64_t amgb_matrix_stream_bytes(amgb_matrix* A, int kind) {
  if (!A) return -1;
  if (kind != 1) return A->op.rows_of_A().stored_bytes();
  int64_t total = 0;
  for (auto& c : A->op.color_sell) total += c->stored_bytes();
  return total;
}

// ---- hierarchy ----
void amgb_options_default(amgb_options* opt) {
  if (opt) options_default(opt);
}

// ---- device-side setup helpers (setup_dia.cuh) ----
// A whole level in DIA on the device plus what the host needs to know about it.
struct FullLevel {
  DevDia dia;            // rows of A
  std::vector<int> off;  // kept offsets, ascending
};
// Statistics of a freshly built DIA level, pruning of its empty diagonals, slice masks and the
// DIA-vs-SELL rule of build_dia (host_setup.cpp).  Returns false when diagonal storage would stream
// >25 % more bytes than SELL: the caller falls back to the host setup.
static bool finalize_full_level(FullLevel& F, DevBuf<double>&& val_in, const std::vector<int>& off_in, int n, int ld,
                                cudaStream_t s) {
  DevBuf<double> val = std::move(val_in);
  std::vector<int> off = off_in;
  DevBuf<unsigned long long> count;
  DevBuf<unsigned short> mask;
  std::vector<unsigned long long> hc;
  for (int pass = 0; pass < 2; ++pass) {
    const int nd = (int)off.size();
    count.alloc(nd + 1);
    count.zero(s);
    mask.alloc(std::max(ld / 32, 1));
    if (n > 0) LAUNCH(setup::k_dia_stats, blocks_for(ld, 256), 256, 0, s, val.p, n, ld, nd, count.p, mask.p);
    hc.assign(nd + 1, 0);
    CUDA_CHECK(cudaMemcpyAsync(hc.data(), count.p, (nd + 1) * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
    CUDA_CHECK(cudaStreamSynchronize(s));
    int kept = 0;
    for (int d = 0; d < nd; ++d) kept += hc[d] != 0;
    if (kept == nd) break;
    // drop the diagonals without an entry (explicit zeros only): the host layout has none either
    DevBuf<double> packed;
    packed.alloc((size_t)std::max(kept, 1) * ld);
    std::vector<int> off2;
    for (int d = 0; d < nd; ++d)
      if (hc[d] != 0) {
        CUDA_CHECK(cudaMemcpyAsync(packed.p + (size_t)off2.size() * ld, val.p + (size_t)d * ld, sizeof(double) * ld,
                                   cudaMemcpyDeviceToDevice, s));
        off2.push_back(off[d]);
      }
    CUDA_CHECK(cudaStreamSynchronize(s));
    val = std::move(packed);
    off = off2;
  }
  const int nd = (int)off.size();
  int64_t nnz = 0;
  for (int d = 0; d < nd; ++d) nnz += (int64_t)hc[d];
  if (8.0 * nd * ld > 1.25 * 12.0 * (double)nnz + 4096.0) return false;
  DevDia& D = F.dia;
  D.n_rows = n;
  D.c_min = 0;
  D.c_max = n - 1;
  D.ld = ld;
  D.n_diag = nd;
  D.nnz = nnz;
  for (int d = 0; d < nd; ++d) D.off[d] = off[d];
  D.live_bytes = (int64_t)nd * ld * 8;
  const int64_t live = (int64_t)hc[nd], n_slices = ld / 32;
  if (live * 10 <= (int64_t)nd * n_slices * 9) {  // skipping empty slices saves >= a tenth of the matrix bytes
    D.mask = std::move(mask);
    D.live_bytes = n_slices * 2 + 256ll * live;
  }
  D.val = std::move(val);
  F.off = off;
  return true;
}
// Rows [row_begin, row_begin + n_dst) of a whole-level DIA with local numbering (rows outside the
// level stay empty); with_stats: also the slice masks and entry count (the per-operator kernels use them).
static void slice_level(const FullLevel& F, int n_src, int row_begin, int n_dst, DevDia& out, bool with_stats,
                        cudaStream_t s) {
  const int nd = F.dia.n_diag;
  const int ld = (n_dst + 31) / 32 * 32;
  out.val.alloc((size_t)std::max(nd, 1) * std::max(ld, 32));
  out.val.zero(s);
  if (n_dst > 0)
    LAUNCH(setup::k_dia_slice, blocks_for(n_dst, 256), 256, 0, s, F.dia.val.p, n_src, F.dia.ld, nd, row_begin, out.val.p,
           n_dst, ld);
  out.n_rows = n_dst;
  out.c_min = 0;
  out.c_max = n_src - 1;
  out.ld = ld;
  out.n_diag = nd;
  for (int d = 0; d < nd; ++d) out.off[d] = F.dia.off[d];
  out.live_bytes = (int64_t)nd * ld * 8;
  out.nnz = 0;
  if (with_stats && n_dst > 0) {
    DevBuf<unsigned long long> count;
    count.alloc(nd + 1);
    count.zero(s);
    DevBuf<unsigned short> mask;
    mask.alloc(std::max(ld / 32, 1));
    LAUNCH(setup::k_dia_stats, blocks_for(ld, 256), 256, 0, s, out.val.p, n_dst, ld, nd, count.p, mask.p);
    std::vector<unsigned long long> hc(nd + 1, 0);
    CUDA_CHECK(cudaMemcpyAsync(hc.data(), count.p, (nd + 1) * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
    CUDA_CHECK(cudaStreamSynchronize(s));
    for (int d = 0; d < nd; ++d) out.nnz += (int64_t)hc[d];
    const int64_t live = (int64_t)hc[nd], n_slices = ld / 32;
    if (live * 10 <= (int64_t)nd * n_slices * 9) {
      out.mask = std::move(mask);
      out.live_bytes = n_slices * 2 + 256ll * live;
    }
  }
}
// ---- device-side smoothed-aggregation setup (setup_sa.cuh) ----
// Exclusive prefix sum of c[0..n) into out[0..n] (out[n] = total), returned.
static int64_t exclusive_scan(const long long* c, int64_t n, DevBuf<long long>& out, cudaStream_t s) {
  out.alloc((size_t)n + 1);
  out.zero(s);
  if (n > 0) {
    size_t bytes = 0;
    CUDA_CHECK(cub::DeviceScan::InclusiveSum(nullptr, bytes, c, out.p + 1, n, s));
    DevBuf<unsigned char> tmp;
    tmp.alloc(bytes);
    CUDA_CHECK(cub::DeviceScan::InclusiveSum(tmp.p, bytes, c, out.p + 1, n, s));
  }
  long long total = 0;
  CUDA_CHECK(cudaMemcpyAsync(&total, out.p + n, sizeof(long long), cudaMemcpyDeviceToHost, s));
  CUDA_CHECK(cudaStreamSynchronize(s));
  return total;
}
// int32 column pointers from the entry counts of n columns; overflow_error(what) beyond int32 indexing
static int64_t counts_to_colptr(const long long* c, int64_t n, DevBuf<int>& colptr, const char* what, cudaStream_t s) {
  DevBuf<long long> off;
  const int64_t total = exclusive_scan(c, n, off, s);
  if (total > (int64_t)std::numeric_limits<int>::max()) throw std::overflow_error(what);
  colptr.alloc((size_t)n + 1);
  LAUNCH(sasetup::k_narrow<int>, blocks_for(n + 1, 256), 256, 0, s, off.p, colptr.p, n + 1);
  return total;
}

// T = A^T, entries of a column in ascending row (a stable sort of the entries by row; host: transpose)
static void dev_transpose(const DevCsc& A, DevCsc& T, cudaStream_t s) {
  const int64_t nnz = A.nnz;
  T.rows = A.cols;
  T.cols = A.rows;
  T.nnz = nnz;
  DevBuf<long long> counts;
  counts.alloc((size_t)A.rows + 1);
  counts.zero(s);
  T.rowidx.alloc(nnz);
  T.val.alloc(nnz);
  if (nnz > 0) {
    DevBuf<int> col_of, perm_in, perm, keys;
    col_of.alloc(nnz);
    perm_in.alloc(nnz);
    perm.alloc(nnz);
    keys.alloc(nnz);
    LAUNCH(sasetup::k_col_of, blocks_for(A.cols, 256), 256, 0, s, A.colptr.p, A.cols, col_of.p);
    LAUNCH(sasetup::k_iota, blocks_for(nnz, 256), 256, 0, s, perm_in.p, nnz);
    LAUNCH(sasetup::k_row_count, blocks_for(nnz, 256), 256, 0, s, A.rowidx.p, nnz, counts.p);
    int end_bit = 1;
    while (end_bit < 31 && (1ll << end_bit) < (long long)A.rows) ++end_bit;
    size_t bytes = 0;
    CUDA_CHECK(cub::DeviceRadixSort::SortPairs(nullptr, bytes, A.rowidx.p, keys.p, perm_in.p, perm.p, (int)nnz, 0,
                                               end_bit, s));
    DevBuf<unsigned char> tmp;
    tmp.alloc(bytes);
    CUDA_CHECK(cub::DeviceRadixSort::SortPairs(tmp.p, bytes, A.rowidx.p, keys.p, perm_in.p, perm.p, (int)nnz, 0, end_bit,
                                               s));
    LAUNCH(sasetup::k_transpose_gather, blocks_for(nnz, 256), 256, 0, s, perm.p, col_of.p, A.val.p, nnz, T.rowidx.p,
           T.val.p);
  }
  counts_to_colptr(counts.p, A.rows, T.colptr, "transpose: exceeds int32 indexing", s);
}

// bitwise_equal on the device
static bool dev_equal(const DevCsc& A, const DevCsc& B, cudaStream_t s) {
  if (A.rows != B.rows || A.cols != B.cols || A.nnz != B.nnz) return false;
  DevBuf<int> flag;
  flag.alloc(1);
  flag.zero(s);
  LAUNCH(sasetup::k_bits_differ<int>, blocks_for(A.cols + 1, 256), 256, 0, s, A.colptr.p, B.colptr.p, A.cols + 1, flag.p);
  if (A.nnz > 0) {
    LAUNCH(sasetup::k_bits_differ<int>, blocks_for(A.nnz, 256), 256, 0, s, A.rowidx.p, B.rowidx.p, A.nnz, flag.p);
    LAUNCH(sasetup::k_bits_differ<double>, blocks_for(A.nnz, 256), 256, 0, s, A.val.p, B.val.p, A.nnz, flag.p);
  }
  int differ = 0;
  CUDA_CHECK(cudaMemcpyAsync(&differ, flag.p, sizeof(int), cudaMemcpyDeviceToHost, s));
  CUDA_CHECK(cudaStreamSynchronize(s));
  return !differ;
}

// C = L R in Eigen's conservative order (host: multiply; plus_zero: the sums start from +0).  what: the
// overflow_error message when C exceeds int32 indexing.
static void dev_multiply(const DevCsc& L, const DevCsc& R, DevCsc& C, bool plus_zero, const char* what, cudaStream_t s) {
  if (L.cols != R.rows) throw std::invalid_argument("multiply: inner dimensions differ");
  const int n = R.cols;
  C.rows = L.rows;
  C.cols = n;
  DevBuf<long long> bound, count;
  DevBuf<int> big, n_big;
  DevBuf<unsigned long long> max_big;
  bound.alloc(n);
  count.alloc(n);
  big.alloc(n);
  n_big.alloc(1);
  n_big.zero(s);
  max_big.alloc(1);
  max_big.zero(s);
  if (n > 0)
    LAUNCH(sasetup::k_spgemm_bound, blocks_for(n, 256), 256, 0, s, L.view(), R.view(), bound.p,
           (long long)sasetup::kSmallSlots / 2, big.p, n_big.p, max_big.p);
  int hb = 0;
  unsigned long long hmax = 0;
  CUDA_CHECK(cudaMemcpyAsync(&hb, n_big.p, sizeof(int), cudaMemcpyDeviceToHost, s));
  CUDA_CHECK(cudaMemcpyAsync(&hmax, max_big.p, sizeof(hmax), cudaMemcpyDeviceToHost, s));
  CUDA_CHECK(cudaStreamSynchronize(s));
  // columns whose table exceeds the shared slots: per-warp tables in global memory, at most ~1 GB of them
  int g_slots = 32;
  while ((unsigned long long)g_slots < 2 * hmax) g_slots <<= 1;
  const int64_t slot_bytes = (int64_t)g_slots * (sizeof(int) + sizeof(double));
  const int64_t g_warps = std::max<int64_t>(1, std::min<int64_t>(hb, (1ll << 30) / slot_bytes));
  const int g_blocks = blocks_for(g_warps, sasetup::kSpgemmWarps);
  DevBuf<int> g_keys;
  DevBuf<double> g_vals;
  if (hb > 0) {
    g_keys.alloc((size_t)g_blocks * sasetup::kSpgemmWarps * g_slots);
    g_vals.alloc((size_t)g_blocks * sasetup::kSpgemmWarps * g_slots);
  }
  const int threads = sasetup::kSpgemmWarps * 32;
  const int s_blocks = std::max(1, std::min(blocks_for(n, sasetup::kSpgemmWarps), 8192));
  auto run = [&](auto kern, int* c_rowidx, double* c_val, const long long* cptr) {
    CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sasetup::kSpgemmSmem));
    if (n > 0)
      LAUNCH(kern, s_blocks, threads, sasetup::kSpgemmSmem, s, L.view(), R.view(), bound.p, nullptr, 0, nullptr,
             nullptr, 0, count.p, cptr, c_rowidx, c_val);
    if (hb > 0)
      LAUNCH(kern, g_blocks, threads, 0, s, L.view(), R.view(), bound.p, big.p, hb, g_keys.p, g_vals.p, g_slots,
             count.p, cptr, c_rowidx, c_val);
  };
  // symbolic pass: entries per column
  run(sasetup::k_spgemm<false, false>, nullptr, nullptr, nullptr);
  DevBuf<long long> off;
  const int64_t total = exclusive_scan(count.p, n, off, s);
  if (total > (int64_t)std::numeric_limits<int>::max()) throw std::overflow_error(what);
  C.nnz = total;
  C.colptr.alloc((size_t)n + 1);
  LAUNCH(sasetup::k_narrow<int>, blocks_for((int64_t)n + 1, 256), 256, 0, s, off.p, C.colptr.p, (int64_t)n + 1);
  // numeric pass (unsorted columns), then every column sorted by row
  DevBuf<int> rowidx_u;
  DevBuf<double> val_u;
  rowidx_u.alloc(total);
  val_u.alloc(total);
  if (plus_zero) run(sasetup::k_spgemm<true, true>, rowidx_u.p, val_u.p, off.p);
  else run(sasetup::k_spgemm<true, false>, rowidx_u.p, val_u.p, off.p);
  C.rowidx.alloc(total);
  C.val.alloc(total);
  if (total > 0) {
    size_t bytes = 0;
    CUDA_CHECK(cub::DeviceSegmentedSort::SortPairs(nullptr, bytes, rowidx_u.p, C.rowidx.p, val_u.p, C.val.p, (int)total,
                                                   n, C.colptr.p, C.colptr.p + 1, s));
    DevBuf<unsigned char> tmp;
    tmp.alloc(bytes);
    CUDA_CHECK(cub::DeviceSegmentedSort::SortPairs(tmp.p, bytes, rowidx_u.p, C.rowidx.p, val_u.p, C.val.p, (int)total, n,
                                                   C.colptr.p, C.colptr.p + 1, s));
  }
  CUDA_CHECK(cudaStreamSynchronize(s));
}

// build_sell of a device CSC ("row c = CSC column c", explicit zeros dropped), on the device
static void dev_sell(const DevCsc& M, DevSell& S, cudaStream_t s) {
  const int n = M.cols;
  const int n_slices = (n + 31) / 32;
  DevBuf<int> len;
  DevBuf<unsigned long long> nnz;
  DevBuf<long long> size;
  len.alloc(n);
  nnz.alloc(1);
  nnz.zero(s);
  size.alloc(n_slices);
  if (n > 0) {
    LAUNCH(sasetup::k_sell_len, blocks_for(n, 256), 256, 0, s, M.view(), len.p, nnz.p);
    LAUNCH(sasetup::k_sell_slice_size, blocks_for(n, 256), 256, 0, s, len.p, n, size.p);
  }
  DevBuf<long long> off;
  const int64_t total = exclusive_scan(size.p, n_slices, off, s);
  if (total > 0xffffffffll) throw std::overflow_error("SELL layout exceeds 32-bit offsets");
  S.n_rows = n;
  S.n_slices = n_slices;
  S.slice_ptr.alloc((size_t)n_slices + 1);
  LAUNCH(sasetup::k_narrow<uint32_t>, blocks_for((int64_t)n_slices + 1, 256), 256, 0, s, off.p, S.slice_ptr.p,
         (int64_t)n_slices + 1);
  S.col.alloc(total);
  S.val.alloc(total);
  CUDA_CHECK(cudaMemsetAsync(S.col.p, 0xff, std::max<int64_t>(total, 1) * sizeof(int), s));
  S.val.zero(s);
  S.rows.release();
  if (n > 0) LAUNCH(sasetup::k_sell_fill, blocks_for(n, 256), 256, 0, s, M.view(), off.p, S.col.p, S.val.p);
  unsigned long long hn = 0;
  CUDA_CHECK(cudaMemcpyAsync(&hn, nnz.p, sizeof(hn), cudaMemcpyDeviceToHost, s));
  CUDA_CHECK(cudaStreamSynchronize(s));
  S.nnz = (int64_t)hn;
}

// build_dia of a square device CSC on the device; false where build_dia refuses (more than 16 offsets, or
// diagonal storage streaming > 25 % more bytes than SELL)
static bool dev_dia(const DevCsc& M, DevDia& D, cudaStream_t s) {
  const int n = M.cols;
  if (n < 1 || M.rows != n) return false;
  const int shift = n - 1;
  const int n_words = (2 * n - 1 + 31) / 32;
  DevBuf<unsigned> bitmap;
  bitmap.alloc(n_words);
  bitmap.zero(s);
  DevBuf<int> list;
  list.alloc(2 + setup::kMaxOffsets);
  list.zero(s);
  LAUNCH(sasetup::k_mark_offsets_nz, blocks_for(n, 256), 256, 0, s, M.view(), shift, bitmap.p);
  LAUNCH(setup::k_collect_offsets, blocks_for(n_words, 256), 256, 0, s, bitmap.p, n_words, shift, setup::kMaxOffsets,
         list.p);
  std::vector<int> hl(2 + setup::kMaxOffsets, 0);
  CUDA_CHECK(cudaMemcpyAsync(hl.data(), list.p, hl.size() * sizeof(int), cudaMemcpyDeviceToHost, s));
  CUDA_CHECK(cudaStreamSynchronize(s));
  if (hl[0] < 1 || hl[0] > setup::kMaxOffsets) return false;
  std::vector<int> off(hl.begin() + 1, hl.begin() + 1 + hl[0]);
  std::sort(off.begin(), off.end());
  setup::Offsets o{};
  o.n = (int)off.size();
  for (int d = 0; d < o.n; ++d) o.v[d] = off[d];
  const int ld = (n + 31) / 32 * 32;
  DevBuf<double> val;
  val.alloc((size_t)off.size() * ld);
  val.zero(s);
  LAUNCH(sasetup::k_csc_to_dia_nz, blocks_for(n, 256), 256, 0, s, M.colptr.p, M.rowidx.p, M.val.p, n, o, val.p, ld);
  FullLevel F;
  if (!finalize_full_level(F, std::move(val), off, n, ld, s)) return false;
  D = std::move(F.dia);
  return true;
}

// DevMat::upload of a device CSC: DIA when build_dia accepts it, else SELL-32
static void dev_mat(const DevCsc& M, DevMat& out, cudaStream_t s) {
  out.is_dia = dev_dia(M, out.dia, s);
  if (!out.is_dia) dev_sell(M, out.sell, s);
}

// sa_hierarchy on the device: A[0] = the level-0 operator, then P[l], R[l] = P[l]^T and A[l + 1] = R (A P)
// while the hierarchy grows (same stop rule, same errors).  The strong graph of every level is downloaded
// and aggregated on the host by the same passes as sa_aggregate.  phase_s accumulates the seconds of
// [strength + aggregation, prolongators, Galerkin products], each phase ending in a stream synchronise.
static void sa_device_hierarchy(int n_levels, double theta, std::vector<DevCsc>& A, std::vector<DevCsc>& P,
                                std::vector<DevCsc>& R, double* phase_s, cudaStream_t s) {
  using clock = std::chrono::steady_clock;
  auto lap = [&](clock::time_point& t0, int phase) {
    CUDA_CHECK(cudaStreamSynchronize(s));
    const clock::time_point t1 = clock::now();
    phase_s[phase] += std::chrono::duration<double>(t1 - t0).count();
    t0 = t1;
  };
  P.clear();
  R.clear();
  while ((int)A.size() < n_levels && A.back().cols > kSaMaxCoarse) {
    const int l = (int)A.size() - 1;
    const int n = A[l].cols;
    const sasetup::CscView M = A[l].view();
    clock::time_point t0 = clock::now();
    // diagonal and strength graph
    DevBuf<double> d;
    d.alloc(n);
    DevBuf<int> zero_row;
    const int none = std::numeric_limits<int>::max();
    zero_row.upload(&none, 1, s);
    LAUNCH(sasetup::k_sa_diag, blocks_for(n, 256), 256, 0, s, M, d.p, zero_row.p);
    int zr = none;
    CUDA_CHECK(cudaMemcpyAsync(&zr, zero_row.p, sizeof(int), cudaMemcpyDeviceToHost, s));
    CUDA_CHECK(cudaStreamSynchronize(s));
    if (zr != none) throw std::invalid_argument(sa_zero_diagonal_message(l, zr));
    DevBuf<long long> cnt, sptr;
    cnt.alloc(n);
    LAUNCH(sasetup::k_sa_strength<false>, blocks_for(n, 256), 256, 0, s, M, d.p, theta, cnt.p, nullptr, nullptr);
    const int64_t n_strong = exclusive_scan(cnt.p, n, sptr, s);
    DevBuf<int> snb, sptr32;
    snb.alloc(n_strong);
    sptr32.alloc((size_t)n + 1);
    LAUNCH(sasetup::k_sa_strength<true>, blocks_for(n, 256), 256, 0, s, M, d.p, theta, nullptr, sptr.p, snb.p);
    LAUNCH(sasetup::k_narrow<int>, blocks_for((int64_t)n + 1, 256), 256, 0, s, sptr.p, sptr32.p, (int64_t)n + 1);
    std::vector<int> h_sptr((size_t)n + 1), h_snb((size_t)n_strong);
    sptr32.download(h_sptr.data(), s);
    snb.download(h_snb.data(), s);
    CUDA_CHECK(cudaStreamSynchronize(s));
    std::vector<int> agg;
    const int64_t n_agg = sa_aggregate_passes(n, h_sptr.data(), h_snb.data(), agg);
    if (n_agg >= n) {
      if (l == 0) throw std::invalid_argument(sa_no_reduction_message(n, n_agg));
      break;
    }
    DevCsc T;  // aggregate indicator, transposed: column k holds (agg[k], 1.0)
    T.rows = (int)n_agg;
    T.cols = n;
    T.nnz = n;
    T.rowidx.upload(agg, s);
    T.colptr.alloc((size_t)n + 1);
    T.val.alloc(n);
    LAUNCH(sasetup::k_iota, blocks_for((int64_t)n + 1, 256), 256, 0, s, T.colptr.p, (int64_t)n + 1);
    LAUNCH(sasetup::k_fill, blocks_for(n, 256), 256, 0, s, T.val.p, n, 1.0);
    lap(t0, 0);
    // smoothed prolongator, built as R = P^T: S = T A sums the entries of every row i per aggregate, then
    // R(J, i) = (J == agg[i]) - (w / a_ii) S(J, i)
    DevBuf<unsigned long long> rho_bits;
    rho_bits.alloc(1);
    rho_bits.zero(s);
    LAUNCH(sasetup::k_sa_gershgorin, blocks_for(n, 256), 256, 0, s, M, d.p, rho_bits.p);
    unsigned long long rb = 0;
    CUDA_CHECK(cudaMemcpyAsync(&rb, rho_bits.p, sizeof(rb), cudaMemcpyDeviceToHost, s));
    CUDA_CHECK(cudaStreamSynchronize(s));
    double rho;
    std::memcpy(&rho, &rb, sizeof(rho));
    const double w = (4.0 / 3.0) / rho;
    DevCsc Rl, Pl;
    dev_multiply(T, A[l], Rl, true, "sa_prolongation: P exceeds int32 indexing", s);
    LAUNCH(sasetup::k_sa_smooth, blocks_for(n, 256), 256, 0, s, n, Rl.colptr.p, Rl.rowidx.p, Rl.val.p, T.rowidx.p, d.p, w);
    dev_transpose(Rl, Pl, s);
    lap(t0, 1);
    // Galerkin product A_{l+1} = R (A P)
    DevCsc AP, AH;
    dev_multiply(A[l], Pl, AP, false, "multiply: result exceeds int32 indexing", s);
    dev_multiply(Rl, AP, AH, false, "multiply: result exceeds int32 indexing", s);
    lap(t0, 2);
    P.push_back(std::move(Pl));
    R.push_back(std::move(Rl));
    A.push_back(std::move(AH));
  }
}

// The whole hierarchy on the device: level 0 from the raw CSC arrays, levels >= 1 by Galerkin products.
// false: the operator (or one of its coarse operators) does not fit the DIA layout -> host setup.
static bool device_build_levels(amgb_hierarchy* h, int n_rows, const int* colptr, const int* rowidx, const double* val,
                                std::vector<FullLevel>& full) {
  cudaStream_t s = h->stream;
  const int L = h->L;
  const int64_t nnz = colptr[n_rows];
  if (n_rows < 1 || nnz < 1) return false;
  if (h->bilinear()) {
    // the row-wise 2-D product needs a 3 x 3 grid stencil (every level below is one then); anything
    // else is left to the host product
    // entry (r, c) couples grid point c = (y, x) to r = c + d: allowed are d = dy m + dx with dy, dx in
    // {-1, 0, 1} and x + dx inside the line (no entry across a line end); x is tracked, not divided out
    const int m = (int)h->m[0];
    if (m < 3) return false;
    for (int c = 0, x = 0; c < n_rows; ++c, x = (x + 1 == m) ? 0 : x + 1)
      for (int p = colptr[c]; p < colptr[c + 1]; ++p) {
        if (val[p] == 0.0) continue;
        const int d = rowidx[p] - c;
        const int dy = (d > 1) ? 1 : (d < -1 ? -1 : 0);
        const int dx = d - dy * m;
        if (dx < -1 || dx > 1 || x + dx < 0 || x + dx >= m) return false;
      }
  }
  h->raw_rows = n_rows;
  h->raw_colptr.upload(colptr, (size_t)n_rows + 1, s);
  h->raw_rowidx.upload(rowidx, (size_t)nnz, s);
  h->raw_val.upload(val, (size_t)nnz, s);
  // distinct offsets
  const int shift = n_rows - 1;
  const int n_words = (2 * n_rows - 1 + 31) / 32;
  DevBuf<unsigned> bitmap;
  bitmap.alloc(n_words);
  bitmap.zero(s);
  DevBuf<int> list;
  list.alloc(2 + setup::kMaxOffsets);
  list.zero(s);
  LAUNCH(setup::k_mark_offsets, blocks_for(n_rows, 256), 256, 0, s, h->raw_colptr.p, h->raw_rowidx.p, n_rows, shift,
         bitmap.p);
  LAUNCH(setup::k_collect_offsets, blocks_for(n_words, 256), 256, 0, s, bitmap.p, n_words, shift, setup::kMaxOffsets,
         list.p);
  std::vector<int> hl(2 + setup::kMaxOffsets, 0);
  CUDA_CHECK(cudaMemcpyAsync(hl.data(), list.p, hl.size() * sizeof(int), cudaMemcpyDeviceToHost, s));
  CUDA_CHECK(cudaStreamSynchronize(s));
  if (hl[0] < 1 || hl[0] > setup::kMaxOffsets) return false;
  std::vector<int> off(hl.begin() + 1, hl.begin() + 1 + hl[0]);
  std::sort(off.begin(), off.end());
  auto pack = [](const std::vector<int>& v) {
    setup::Offsets o{};
    o.n = (int)v.size();
    for (int d = 0; d < o.n; ++d) o.v[d] = v[d];
    return o;
  };
  // DIA of "row c = CSC column c" (rows of A^T), then rows of A (the same array when A is bitwise symmetric)
  const int ld0 = (n_rows + 31) / 32 * 32;
  DevBuf<double> colrows;
  colrows.alloc((size_t)off.size() * ld0);
  colrows.zero(s);
  LAUNCH(setup::k_csc_to_dia, blocks_for(n_rows, 256), 256, 0, s, h->raw_colptr.p, h->raw_rowidx.p, h->raw_val.p, n_rows,
         pack(off), colrows.p, ld0);
  DevBuf<int> flag;
  flag.alloc(1);
  flag.zero(s);
  LAUNCH(setup::k_dia_asymmetric, blocks_for(n_rows, 256), 256, 0, s, colrows.p, n_rows, ld0, pack(off), flag.p);
  int asym = 0;
  CUDA_CHECK(cudaMemcpyAsync(&asym, flag.p, sizeof(int), cudaMemcpyDeviceToHost, s));
  CUDA_CHECK(cudaStreamSynchronize(s));
  full.clear();
  full.resize(L);
  if (asym) {
    std::vector<int> off_t;
    for (auto it = off.rbegin(); it != off.rend(); ++it) off_t.push_back(-*it);
    DevBuf<double> rowsA;
    rowsA.alloc((size_t)off_t.size() * ld0);
    rowsA.zero(s);
    LAUNCH(setup::k_dia_transpose, blocks_for(n_rows, 256), 256, 0, s, colrows.p, n_rows, ld0, pack(off), pack(off_t),
           rowsA.p);
    if (!finalize_full_level(full[0], std::move(rowsA), off_t, n_rows, ld0, s)) return false;
  } else {
    if (!finalize_full_level(full[0], std::move(colrows), off, n_rows, ld0, s)) return false;
  }
  // coarse levels: A_{l+1} = R (A_l P), one thread per coarse row (multigrid.hpp:219-223)
  for (int l = 1; l < L; ++l) {
    const int n_f = (int)h->n[l - 1], n_c = (int)h->n[l];
    const DevDia& Fd = full[l - 1].dia;
    gal::FineDia A;
    A.n = n_f;
    A.nd = Fd.n_diag;
    A.ld = Fd.ld;
    for (int d = 0; d < A.nd; ++d) A.off[d] = Fd.off[d];
    A.val = Fd.val.p;
    CoarseOffsets oc{};
    const int nd_c = h->bilinear() ? gal::coarse_offsets_2d((int)h->m[l], oc.v) : gal::coarse_offsets(A.nd, A.off, oc.v);
    if (nd_c < 1) return false;
    const int ld_c = (n_c + 31) / 32 * 32;
    DevBuf<double> out;
    out.alloc((size_t)nd_c * ld_c);
    out.zero(s);
    if (h->bilinear())
      LAUNCH(k_galerkin_dia2d, blocks_for(n_c, 256), 256, 0, s, A, (int)h->m[l - 1], (int)h->m[l], nd_c, oc, out.p, ld_c);
    else
      LAUNCH(k_galerkin_dia, blocks_for(n_c, 256), 256, 0, s, A, n_c, nd_c, oc, out.p, ld_c);
    std::vector<int> off_c(oc.v, oc.v + nd_c);
    if (!finalize_full_level(full[l], std::move(out), off_c, n_c, ld_c, s)) return false;
  }
  return true;
}
// host CSC (rows of A, explicit zeros already dropped) of a small device DIA level: the coarsest factorisation
static Csc csc_from_device_dia(const DevDia& D, cudaStream_t s) {
  std::vector<double> v((size_t)D.n_diag * D.ld);
  CUDA_CHECK(cudaMemcpyAsync(v.data(), D.val.p, v.size() * sizeof(double), cudaMemcpyDeviceToHost, s));
  CUDA_CHECK(cudaStreamSynchronize(s));
  // assemble row by row (column k of M = row k of A), then transpose: the factorisation reads the lower
  // triangle A(r, c), r >= c, exactly like the host path does for operators symmetric only up to rounding
  Csc M;
  M.rows = M.cols = D.n_rows;
  M.colptr.assign((size_t)D.n_rows + 1, 0);
  for (int r = 0; r < D.n_rows; ++r) {
    for (int d = 0; d < D.n_diag; ++d) {
      const double a = v[(size_t)d * D.ld + r];
      const int c = r + D.off[d];
      if (a != 0.0 && c >= 0 && c < D.n_rows) {
        M.rowidx.push_back(c);
        M.val.push_back(a);
      }
    }
    M.colptr[(size_t)r + 1] = (int)M.rowidx.size();
  }
  return transpose(M);  // columns of A, like the host path's mats[L - 1]
}

static void create_hierarchy(amgb_comm* comm, int64_t min_rows_per_rank, int n_rows, int n_cols,
                             const int* colptr, const int* rowidx, const double* val, const double* b,
                             int64_t b_rows, const amgb_options* opt_in, amgb_hierarchy** out) {
  if (!out || !opt_in || !colptr) throw std::invalid_argument("null argument");
  const amgb_options& o = *opt_in;
  // multigrid.hpp:165-178 -- same order, same messages
  if (o.compute_error_every_n_iters > o.n_iters)
    throw std::invalid_argument("`compute_error_every_n_iters` must be leq to `n_iters`, got " +
                                std::to_string(o.compute_error_every_n_iters) + " and " +
                                std::to_string(o.n_iters));
  if ((int64_t)n_rows != b_rows)
    throw std::invalid_argument("`A` and `b` must have the same number of degrees of freedom, got " +
                                std::to_string(n_rows) + " and " + std::to_string(b_rows));
  if (o.n_levels < 1) throw std::invalid_argument("n_levels must be >= 1");
  if (n_rows != n_cols) throw std::invalid_argument("A must be square");
  if (o.smoother < 0 || o.smoother > 3) throw std::invalid_argument("unknown smoother kind");
  if (o.arith != AMGB_ARITH_REFERENCE && o.arith != AMGB_ARITH_FAST) throw std::invalid_argument("unknown arithmetic mode");
  if (o.transfer != AMGB_TRANSFER_LINEAR && o.transfer != AMGB_TRANSFER_BILINEAR_2D &&
      o.transfer != AMGB_TRANSFER_SMOOTHED_AGGREGATION)
    throw std::invalid_argument("unknown transfer kind");
  if (o.transfer == AMGB_TRANSFER_SMOOTHED_AGGREGATION) {
    if (!(o.strength >= 0.0))
      throw std::invalid_argument("smoothed aggregation: strength must be >= 0, got " + std::to_string(o.strength));
    if (comm)
      throw std::invalid_argument("smoothed aggregation has no sharded hierarchy: aggregate numbering does not give "
                                  "row blocks whose halos come from ranks +-1 only (use amgb_hierarchy_create)");
  }
  if (o.transfer == AMGB_TRANSFER_BILINEAR_2D) {
    if (grid_lines(n_rows) < 1)
      throw std::invalid_argument("the bilinear 2-D transfer needs an m x m grid operator, got " + std::to_string(n_rows) +
                                  " rows (not a square number)");
  }
  if (o.smoother == AMGB_SMOOTHER_LINE_GS) {
    if (o.lines != AMGB_LINES_X && o.lines != AMGB_LINES_Y && o.lines != AMGB_LINES_ALTERNATING)
      throw std::invalid_argument("unknown line direction setting " + std::to_string(o.lines) +
                                  " (AMGB_LINES_X, AMGB_LINES_Y or AMGB_LINES_ALTERNATING)");
    if (o.transfer != AMGB_TRANSFER_BILINEAR_2D)
      throw std::invalid_argument("line Gauss-Seidel needs the bilinear 2-D transfer (AMGB_TRANSFER_BILINEAR_2D): "
                                  "the coarse levels of the linear and smoothed-aggregation transfers are not grids");
  }
  if (!b || !rowidx || !val) throw std::invalid_argument("null argument");
  require_device();

  std::unique_ptr<amgb_hierarchy> h(new amgb_hierarchy());
  h->opt = o;
  // fuse bits 1-7 (folded prolongation, fused legs, coarse tail, mid levels, compressed formats) hard-code
  // the 1-D transfer; a 2-D hierarchy runs the per-operator cycle with the zero-guess first sweep only
  if (h->bilinear() || h->sa()) h->opt.fuse &= 1;
  h->L = o.n_levels;
  h->comm = comm;
  CUDA_CHECK(cudaGetDevice(&h->device));
  CUDA_CHECK(cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));
  h->stream = h->own_stream;
  cudaStream_t s = h->stream;

  std::vector<Csc> mats;
  const char* force_host = std::getenv("AMGB_HOST_SETUP");
  const bool host_setup = force_host && std::string(force_host) == "1";
  using clock = std::chrono::steady_clock;
  clock::time_point sa_t0 = clock::now();
  std::vector<DevMat> sa_rows;  // rows-of-A mirrors of a device-resident smoothed-aggregation hierarchy
  if (h->sa()) {
    // n_levels is a cap.  Device setup unless AMGB_HOST_SETUP=1: the levels and prolongators are built on
    // the GPU; damped Jacobi keeps them there, the Gauss-Seidel smoothers (whose colourings and schedules
    // need host matrices) download them and continue like the host setup
    if (host_setup) {
      sa_hierarchy(csc_from_arrays(n_rows, n_cols, colptr, rowidx, val), o.strength, o.n_levels, mats, h->sa_P,
                   h->sa_times);
      h->L = (int)mats.size();
      sa_t0 = clock::now();
    } else {
      std::vector<DevCsc> A(1), R;
      A[0].upload(n_rows, n_cols, colptr, rowidx, val, s);
      sa_device_hierarchy(o.n_levels, o.strength, A, h->sa_dev_P, R, h->sa_times, s);
      h->device_setup = true;
      h->L = (int)A.size();
      sa_t0 = clock::now();
      const int L = h->L;
      if (o.smoother == AMGB_SMOOTHER_JACOBI) {
        h->sa_resident = true;
        // mirrors: the rows of A (A itself when bitwise symmetric), and SELL rows of R and of P
        sa_rows.resize(L);
        for (int l = 0; l < L; ++l) {
          DevCsc AT;
          dev_transpose(A[l], AT, s);
          dev_mat(dev_equal(A[l], AT, s) ? A[l] : AT, sa_rows[l], s);
        }
        for (int l = 0; l + 1 < L; ++l) {
          h->sa_R_rows.emplace_back();
          dev_sell(h->sa_dev_P[l], h->sa_R_rows.back(), s);
          h->sa_P_rows.emplace_back();
          dev_sell(R[l], h->sa_P_rows.back(), s);
        }
        mats.resize(L);
        mats[L - 1] = A[L - 1].download(s);  // the coarsest factorisation and its size check
        h->sa_dev_A = std::move(A);
      } else {
        for (const DevCsc& M : A) mats.push_back(M.download(s));
        for (const DevCsc& M : h->sa_dev_P) h->sa_P.push_back(M.download(s));
        h->sa_dev_P.clear();
      }
    }
  }
  const int L = h->L;

  // ---- level sizes (multigrid.hpp:127-130, :213-215) ----
  h->n.resize(L);
  h->n[0] = n_rows;
  if (h->bilinear()) h->m.assign(1, grid_lines(n_rows));
  for (int l = 1; l < L; ++l) {
    if (h->sa()) {
      h->n[l] = h->sa_resident ? h->sa_dev_A[l].cols : mats[l].cols;
      continue;
    }
    if (h->bilinear()) {
      h->m.push_back(coarse_lines_2d(h->m[l - 1]));
      h->n[l] = h->m[l] * h->m[l];
    } else {
      h->n[l] = coarse_dofs(h->n[l - 1]);
    }
    if (h->n[l] < 1) throw std::invalid_argument("too many levels: level " + std::to_string(l) + " is empty");
  }

  // ---- the level operators (multigrid.hpp:190-223) ----
  // Damped-Jacobi cycles on banded operators: built on the DEVICE from the raw CSC arrays
  // (setup_dia.cuh); every rank builds the whole (cheap) hierarchy and slices its row blocks.
  // Everything else (Gauss-Seidel schedules and colourings need the host matrices; unstructured
  // operators need SELL): host setup, every rank builds all of it.  AMGB_HOST_SETUP=1 forces the latter.
  std::vector<FullLevel> full;
  if ((o.smoother == AMGB_SMOOTHER_JACOBI || o.smoother == AMGB_SMOOTHER_LINE_GS) && !h->sa() && !host_setup)
    h->device_setup = device_build_levels(h.get(), n_rows, colptr, rowidx, val, full);
  const bool dia_setup = h->device_setup && !h->sa();  // levels built by device_build_levels
  if (!h->device_setup && !h->sa()) {
    full.clear();
    h->raw_colptr.release();
    h->raw_rowidx.release();
    h->raw_val.release();
    mats.resize(L);
    mats[0] = csc_from_arrays(n_rows, n_cols, colptr, rowidx, val);
    for (int l = 1; l < L; ++l) {
      Csc P = h->prolongation(l - 1);
      Csc R = transpose(P);
      mats[l] = galerkin(R, mats[l - 1], P);
    }
  }
  // offsets (col - row of the non-zero entries) of every level, at most 17 kept: half-bandwidths and
  // the line structure the streaming legs need
  std::vector<std::vector<int>> level_off(L);
  std::vector<int> half_bw(L, 0);
  for (int l = 0; l < L; ++l) {
    if (dia_setup) {
      level_off[l] = full[l].off;
    } else {
      const Csc& M = mats[l];
      std::vector<int>& offs = level_off[l];
      for (int c = 0; c < M.cols; ++c)
        for (int p = M.colptr[c]; p < M.colptr[c + 1]; ++p) {
          if (M.val[p] == 0.0) continue;
          const int off = M.rowidx[p] - c;
          half_bw[l] = std::max(half_bw[l], std::abs(off));
          if (offs.size() > 16) continue;
          auto it = std::lower_bound(offs.begin(), offs.end(), off);
          if (it == offs.end() || *it != off) offs.insert(it, off);
        }
    }
    for (int off : level_off[l]) half_bw[l] = std::max(half_bw[l], std::abs(off));
  }
  // coarsest factorisation (multigrid.hpp:240-243); the direct solve is a banded
  // substitution in one block, so refuse hierarchies whose coarsest level is not small
  {
    const int64_t nc = h->n[L - 1], bw = std::max(half_bw[L - 1], 1);
    if ((double)nc * bw * bw > 2e10 || nc * bw > (1ll << 27))
      throw std::invalid_argument("coarsest level too large for the direct solve (" + std::to_string(nc) +
                                  " DOF, half-bandwidth " + std::to_string(bw) + "): use more levels");
  }
  h->factor = dia_setup ? factor_banded_ldlt(csc_from_device_dia(full[L - 1].dia, s)) : factor_banded_ldlt(mats[L - 1]);

  // ---- partition (sharded runs only) ----
  const int world = comm ? comm->world : 1;
  if (world > 1) {
    if (o.smoother == AMGB_SMOOTHER_GS)
      throw std::invalid_argument("the row-block sharded V-cycle supports the damped-Jacobi and multicolour "
                                  "Gauss-Seidel smoothers (lexicographic Gauss-Seidel is a single-GPU path)");
    // With the fused legs on, only levels whose operator is a 3 x 3 line stencil are worth
    // sharding (they run as streaming legs on the rank's window); the levels below, a few
    // hundred thousand rows at most, are agglomerated.
    int max_sharded = 1 << 30;
    if ((h->opt.fuse & 4) && o.smoother == AMGB_SMOOTHER_JACOBI && (o.smoother_iters == 1 || o.smoother_iters == 2)) {
      max_sharded = 0;
      for (int l = 0; l + 1 < L; ++l) {
        const std::vector<int>& offs = level_off[l];
        if (offs.empty() || offs.size() > 10) break;
        leg::Plan st = leg::plan_leg(leg::UP, 2, (int)h->n[l], (int)offs.size(), offs.data(), 148, 200 * 1024);
        if (!st.ok || !(st.P.m < st.P.n) || st.P.rho != 1) break;
        unsigned mask = 0;
        for (size_t d = 0; d < offs.size(); ++d) mask |= 1u << ((st.P.line_a[d] + 1) * 3 + st.P.delta[d] + 1);
        if (mask != sleg::kMask5 && mask != sleg::kMask7a && mask != sleg::kMask7b && mask != sleg::kMask9) break;
        max_sharded = l + 1;
      }
      if (max_sharded == 0) max_sharded = 1 << 30;  // no streamable level: the per-operator kernels shard as before
    }
    h->plan = h->bilinear() ? make_partition_plan_2d(h->m, world, min_rows_per_rank)
                            : make_partition_plan(h->n, half_bw, world, min_rows_per_rank, max_sharded);
    h->n_sharded = h->plan.n_sharded;
    if (h->n_sharded > 0) {
      // the first replicated level's rows each rank restricts into: half the fine rows (1-D), or the
      // coarse lines from half the fine block's first line (2-D)
      const int ns = h->n_sharded;
      h->coarse_block_start.resize(world + 1);
      for (int g = 0; g <= world; ++g)
        h->coarse_block_start[g] = (g == world)      ? h->n[ns]
                                   : h->bilinear() ? h->plan.start[ns - 1][g] / h->m[ns - 1] / 2 * h->m[ns]
                                                   : h->plan.start[ns - 1][g] / 2;
    }
  }

  // ---- device mirrors ----
  h->ops.resize(L);
  h->lv.resize(L);
  const int g = comm ? comm->rank : 0;
  for (int l = 0; l < L; ++l) {
    LevelState& S = h->lv[l];
    S.n_global = h->n[l];
    h->ops[l].reset(new Operator());
    const bool want_window =
        (h->opt.fuse & 4) && o.smoother == AMGB_SMOOTHER_JACOBI && (o.smoother_iters == 1 || o.smoother_iters == 2);
    if (l < h->n_sharded) {
      S.sharded = true;
      S.s = h->plan.start[l][g];
      S.e = h->plan.start[l][g + 1];
      S.halo_lo = h->plan.halo_lo[l];
      S.halo_hi = h->plan.halo_hi[l];
      S.n_own = (int)(S.e - S.s);
      S.n_mat = (int)std::min<int64_t>(S.n_own + h->plan.ghost[l], h->n[l] - S.s);
      if (dia_setup) {
        // row block (+ ghost rows) and window of this rank, sliced out of the whole level on the device
        DevDia blk;
        slice_level(full[l], (int)h->n[l], (int)S.s, S.n_mat, blk, true, s);
        blk.c_min = -S.halo_lo;
        blk.c_max = S.n_own + S.halo_hi - 1;
        h->ops[l]->adopt_rows(std::move(blk), S.n_own);
        h->ops[l]->block = true;
        if (want_window) {
          slice_level(full[l], (int)h->n[l], (int)(S.s - S.halo_lo), (int)S.n_vec(), h->ops[l]->win, false, s);
          h->ops[l]->win_off = full[l].off;
        }
        CUDA_CHECK(cudaStreamSynchronize(s));
        full[l].dia.val.release();  // the whole-level copy is not needed any more
        full[l].dia.mask.release();
      } else {
        h->ops[l]->build_block(std::move(mats[l]), (int)S.s, S.n_mat, S.n_own, S.halo_lo, S.halo_hi, s);
      }
    } else {
      S.s = 0;
      S.e = h->n[l];
      S.n_own = S.n_mat = (int)h->n[l];
      if (dia_setup) h->ops[l]->adopt_rows(std::move(full[l].dia), S.n_own);
      else if (h->sa_resident) h->ops[l]->adopt_rows(std::move(sa_rows[l]));
      else h->ops[l]->build(std::move(mats[l]), s);
    }
    // +8: the fused legs copy 16-byte aligned windows, which may reach one entry past the end
    S.u.alloc(S.n_vec() + 8);
    S.u.zero(s);
    S.f.alloc(S.n_mat + 8);
    S.f.zero(s);
    // (sharded: every level vector is exported to the neighbours; smoothed aggregation: the residual goes there)
    if (o.smoother == AMGB_SMOOTHER_JACOBI || S.sharded || h->sa()) {
      S.tmp.alloc(S.n_vec() + 8);
      S.tmp.zero(s);
    }
    if (S.sharded) {
      S.fw.alloc(S.n_vec() + 8);
      S.fw.zero(s);
      // window mirror of the operator for the fused legs (block + ghost rows on both sides)
      if (want_window && !dia_setup) h->ops[l]->build_window((int)(S.s - S.halo_lo), (int)S.n_vec(), s);
    }
    if (!(l + 1 == L && o.skip_dead_coarse_smooth)) h->prepare_smoother(l);
  }
  for (int l = 0; l + 1 < L && h->sa() && !h->sa_resident; ++l) {
    h->sa_R_rows.emplace_back();
    h->sa_R_rows.back().upload(build_sell(h->sa_P[l]), s);
    h->sa_P_rows.emplace_back();
    h->sa_P_rows.back().upload(build_sell(transpose(h->sa_P[l])), s);
  }
  if (h->sa()) {
    CUDA_CHECK(cudaStreamSynchronize(s));
    h->sa_times[3] = std::chrono::duration<double>(clock::now() - sa_t0).count();
  }
  for (int l = 0; l < L; ++l) h->prepare_legs(l);
  {
    // sharded levels hand each other right-hand sides in the window layout: fused legs on all of
    // them or on none
    bool all = true;
    for (int l = 0; l < h->n_sharded; ++l) all = all && h->leg_ok(l);
    if (!all)
      for (int l = 0; l < h->n_sharded; ++l) h->legs[l].ok = false;
  }
  h->upload_f(0, b);
  h->partial.alloc(std::max(1, blocks_for(h->lv[0].n_own, 256)));
  h->scalar.alloc(1);
  h->dL.upload(h->factor.L, s);
  h->dd.upload(h->factor.d, s);
  h->dwork.alloc(h->factor.n);
  CUDA_CHECK(cudaStreamSynchronize(s));
  h->prepare_tail();  // needs the factor on the device
  h->prepare_mid();
  h->setup_p2p();
  *out = h.release();
}

int amgb_hierarchy_create(int n_rows, int n_cols, const int* colptr, const int* rowidx, const double* val,
                          const double* b, int64_t b_rows, const amgb_options* opt_in,
                          amgb_hierarchy** out) {
  return guarded([&] {
    create_hierarchy(nullptr, 0, n_rows, n_cols, colptr, rowidx, val, b, b_rows, opt_in, out);
  });
}
int amgb_hierarchy_create_sharded(amgb_comm* comm, int64_t min_rows_per_rank, int n_rows, int n_cols,
                                  const int* colptr, const int* rowidx, const double* val, const double* b,
                                  int64_t b_rows, const amgb_options* opt_in, amgb_hierarchy** out) {
  return guarded([&] {
    if (!comm) throw std::invalid_argument("null communicator");
    if (opt_in && opt_in->smoother == AMGB_SMOOTHER_LINE_GS)
      throw std::invalid_argument("line Gauss-Seidel is a single-GPU path (no sharded hierarchy): every pass walks "
                                  "whole grid lines, so row blocks would not shorten it");
    if (opt_in && opt_in->transfer == AMGB_TRANSFER_BILINEAR_2D && comm->world < 2)
      throw std::invalid_argument("a sharded bilinear 2-D hierarchy needs a communicator of at least two ranks "
                                  "(nothing to shard: use amgb_hierarchy_create)");
    CUDA_CHECK(cudaSetDevice(comm->device));
    create_hierarchy(comm, std::max<int64_t>(min_rows_per_rank, 1), n_rows, n_cols, colptr, rowidx, val, b,
                     b_rows, opt_in, out);
  });
}
int amgb_hierarchy_n_sharded_levels(const amgb_hierarchy* h) { return h ? h->n_sharded : 0; }
int amgb_hierarchy_local_range(const amgb_hierarchy* h, int level, int64_t* begin, int64_t* end) {
  return guarded([&] {
    if (!h) throw std::invalid_argument("null argument");
    h->check_level(level);
    if (begin) *begin = h->lv[level].s;
    if (end) *end = h->lv[level].e;
  });
}
int64_t amgb_hierarchy_halo_exchanges_per_vcycle(const amgb_hierarchy* h) {
  return h ? h->halo_exchanges_per_vcycle : 0;
}
int amgb_hierarchy_halo_mode(const amgb_hierarchy* h) {
  if (!h || h->n_sharded == 0) return AMGB_HALO_NONE;
  return h->p2p ? AMGB_HALO_PEER : AMGB_HALO_NCCL;
}
int amgb_hierarchy_halo_timed_out(amgb_hierarchy* h) {
  if (!h || !h->timed_out_host) return 0;
  cudaStreamSynchronize(h->stream);
  return *(volatile int*)h->timed_out_host;
}

// ---- communicator ----
int amgb_comm_unique_id_bytes(void) { return (int)sizeof(ncclUniqueId); }
int amgb_comm_get_unique_id(void* id) {
  return guarded([&] {
    if (!id) throw std::invalid_argument("null argument");
    ncclUniqueId u;
    NCCL_CHECK(NcclApi::get().GetUniqueId(&u));
    std::memcpy(id, &u, sizeof(u));
  });
}
int amgb_comm_create(const void* id, int rank, int world, amgb_comm** out) {
  return guarded([&] {
    if (!id || !out || world < 1 || rank < 0 || rank >= world) throw std::invalid_argument("bad communicator arguments");
    require_device();
    std::unique_ptr<amgb_comm> c(new amgb_comm());
    c->rank = rank;
    c->world = world;
    CUDA_CHECK(cudaGetDevice(&c->device));
    ncclUniqueId u;
    std::memcpy(&u, id, sizeof(u));
    NCCL_CHECK(NcclApi::get().CommInitRank(&c->comm, world, u, rank));
    *out = c.release();
  });
}
int amgb_comm_destroy(amgb_comm* c) {
  return guarded([&] {
    if (!c) return;
    cudaSetDevice(c->device);
    delete c;
  });
}
// host-only: the row-block plan a sharded hierarchy would use
int amgb_partition_plan(int n_levels, const int64_t* level_sizes, const int* half_bandwidth, int world,
                        int64_t min_rows_per_rank, int* n_sharded, int64_t* starts, int* halo_lo,
                        int* halo_hi, int* ghost) {
  return guarded([&] {
    if (!level_sizes || !half_bandwidth || !n_sharded || n_levels < 1 || world < 1)
      throw std::invalid_argument("bad plan arguments");
    std::vector<int64_t> sizes(level_sizes, level_sizes + n_levels);
    std::vector<int> bw(half_bandwidth, half_bandwidth + n_levels);
    PartitionPlan P = make_partition_plan(sizes, bw, world, std::max<int64_t>(min_rows_per_rank, 1));
    *n_sharded = P.n_sharded;
    for (int l = 0; l < P.n_sharded; ++l) {
      if (starts)
        for (int g = 0; g <= world; ++g) starts[(size_t)l * (world + 1) + g] = P.start[l][g];
      if (halo_lo) halo_lo[l] = P.halo_lo[l];
      if (halo_hi) halo_hi[l] = P.halo_hi[l];
      if (ghost) ghost[l] = P.ghost[l];
    }
  });
}
int amgb_partition_plan_2d(int n_levels, const int64_t* lines, int world, int64_t min_rows_per_rank, int* n_sharded,
                           int64_t* starts, int* halo_lo, int* halo_hi, int* ghost) {
  return guarded([&] {
    if (!lines || !n_sharded || n_levels < 1 || world < 1) throw std::invalid_argument("bad plan arguments");
    std::vector<int64_t> m(lines, lines + n_levels);
    if (m[0] < 1 || m[0] * m[0] > std::numeric_limits<int>::max())
      throw std::invalid_argument("bad plan arguments: level 0 must have 1 .. 46340 lines");
    for (int l = 1; l < n_levels; ++l)
      if (m[l] < 1 || m[l] != coarse_lines_2d(m[l - 1]))
        throw std::invalid_argument("bad plan arguments: level " + std::to_string(l) + " has " + std::to_string(m[l]) +
                                    " lines, the bilinear transfer gives " + std::to_string(coarse_lines_2d(m[l - 1])));
    PartitionPlan P = make_partition_plan_2d(m, world, std::max<int64_t>(min_rows_per_rank, 1));
    *n_sharded = P.n_sharded;
    for (int l = 0; l < P.n_sharded; ++l) {
      if (starts)
        for (int g = 0; g <= world; ++g) starts[(size_t)l * (world + 1) + g] = P.start[l][g];
      if (halo_lo) halo_lo[l] = P.halo_lo[l];
      if (halo_hi) halo_hi[l] = P.halo_hi[l];
      if (ghost) ghost[l] = P.ghost[l];
    }
  });
}

int amgb_hierarchy_destroy(amgb_hierarchy* h) {
  return guarded([&] {
    if (!h) return;
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    if (h->p2p) {
      // collective: nobody unmaps or frees a vector a neighbour may still write into
      bool ok = true;
      h->stream = h->own_stream;
      h->scalar_host_and(ok);
      for (void* p : h->ipc_opened) cudaIpcCloseMemHandle(p);
      h->ipc_opened.clear();
      h->scalar_host_and(ok);
    }
    delete h;
  });
}
int amgb_hierarchy_set_stream(amgb_hierarchy* h, void* cuda_stream) {
  return guarded([&] {
    if (!h) throw std::invalid_argument("null argument");
    CUDA_CHECK(cudaStreamSynchronize(h->stream));
    h->stream = cuda_stream ? (cudaStream_t)cuda_stream : h->own_stream;
  });
}
int amgb_hierarchy_n_levels(const amgb_hierarchy* h) { return h ? h->L : 0; }
int amgb_hierarchy_transfer(const amgb_hierarchy* h) { return h ? h->opt.transfer : -1; }
int amgb_hierarchy_get_transfer(const amgb_hierarchy* h, int level, int64_t* nnz, int* P_colptr, int* P_rowidx,
                                double* P_val) {
  return guarded([&] {
    if (!h || !nnz) throw std::invalid_argument("null argument");
    h->check_level(level, true);
    const Csc P = h->prolongation(level);
    *nnz = P.nnz();
    if (P_colptr) std::memcpy(P_colptr, P.colptr.data(), P.colptr.size() * sizeof(int));
    if (P_rowidx) std::memcpy(P_rowidx, P.rowidx.data(), P.rowidx.size() * sizeof(int));
    if (P_val) std::memcpy(P_val, P.val.data(), P.val.size() * sizeof(double));
  });
}
// C = A B for host CSC matrices (A: m x k, B: k x n), computed on the device in Eigen's conservative order
// (host_setup.cpp: multiply); the product of the smoothed-aggregation setup
int amgb_csc_multiply(int m, int k, const int* A_colptr, const int* A_rowidx, const double* A_val, int n,
                      const int* B_colptr, const int* B_rowidx, const double* B_val, int64_t* nnz, int* C_colptr,
                      int* C_rowidx, double* C_val) {
  return guarded([&] {
    if (!nnz || !A_colptr || !B_colptr || m < 0 || k < 0 || n < 0) throw std::invalid_argument("bad multiply arguments");
    if (A_colptr[k] > 0 && (!A_rowidx || !A_val)) throw std::invalid_argument("bad multiply arguments");
    if (B_colptr[n] > 0 && (!B_rowidx || !B_val)) throw std::invalid_argument("bad multiply arguments");
    require_device();
    cudaStream_t s = nullptr;
    DevCsc A, B, C;
    A.upload(m, k, A_colptr, A_rowidx, A_val, s);
    B.upload(k, n, B_colptr, B_rowidx, B_val, s);
    dev_multiply(A, B, C, false, "multiply: result exceeds int32 indexing", s);
    *nnz = C.nnz;
    if (C_colptr) C.colptr.download(C_colptr, s);
    if (C_rowidx) C.rowidx.download(C_rowidx, s);
    if (C_val) C.val.download(C_val, s);
    CUDA_CHECK(cudaStreamSynchronize(s));
  });
}

int amgb_hierarchy_device_setup(const amgb_hierarchy* h) { return h && h->device_setup ? 1 : 0; }
int amgb_hierarchy_setup_times(const amgb_hierarchy* h, double* out) {
  return guarded([&] {
    if (!h || !out) throw std::invalid_argument("null argument");
    if (!h->sa()) throw ApiError(AMGB_ESTATE, "setup phase times are recorded for smoothed-aggregation hierarchies only");
    for (int i = 0; i < 4; ++i) out[i] = h->sa_times[i];
  });
}
int64_t amgb_hierarchy_n_dofs(const amgb_hierarchy* h, int level) {
  return (h && level >= 0 && level < h->L) ? h->n[level] : -1;
}
int64_t amgb_hierarchy_nnz(const amgb_hierarchy* h, int level) {
  if (!h || level < 0 || level >= h->L) return -1;
  try {
    if (h->sa_resident) return h->sa_dev_A[level].nnz;
    return const_cast<amgb_hierarchy*>(h)->host_matrix(level).nnz();
  } catch (...) {
    return -1;
  }
}
int64_t amgb_hierarchy_nnz_device(const amgb_hierarchy* h, int level) {
  return (h && level >= 0 && level < h->L) ? h->ops[level]->nnz_device() : -1;
}
double amgb_hierarchy_tolerance(const amgb_hierarchy* h) { return h ? h->opt.tolerance : 0.0; }
int amgb_hierarchy_get_matrix(const amgb_hierarchy* h, int level, int* colptr, int* rowidx, double* val) {
  return guarded([&] {
    if (!h) throw std::invalid_argument("null argument");
    h->check_level(level);
    const Csc& M = const_cast<amgb_hierarchy*>(h)->host_matrix(level);
    if (colptr) std::memcpy(colptr, M.colptr.data(), M.colptr.size() * sizeof(int));
    if (rowidx) std::memcpy(rowidx, M.rowidx.data(), M.rowidx.size() * sizeof(int));
    if (val) std::memcpy(val, M.val.data(), M.val.size() * sizeof(double));
  });
}
int amgb_hierarchy_get_soln(amgb_hierarchy* h, int level, double* u) {
  return guarded([&] {
    if (!h || !u) throw std::invalid_argument("null argument");
    h->check_level(level);
    CUDA_CHECK(cudaSetDevice(h->device));
    h->download(level, true, u);
  });
}
int amgb_hierarchy_get_rhs(amgb_hierarchy* h, int level, double* f) {
  return guarded([&] {
    if (!h || !f) throw std::invalid_argument("null argument");
    h->check_level(level);
    CUDA_CHECK(cudaSetDevice(h->device));
    h->download(level, false, f);
  });
}
int amgb_hierarchy_set_soln(amgb_hierarchy* h, int level, const double* u) {
  return guarded([&] {
    if (!h || !u) throw std::invalid_argument("null argument");
    h->check_level(level);
    CUDA_CHECK(cudaSetDevice(h->device));
    h->upload_u(level, u);
  });
}
int amgb_hierarchy_set_rhs(amgb_hierarchy* h, int level, const double* f) {
  return guarded([&] {
    if (!h || !f) throw std::invalid_argument("null argument");
    h->check_level(level);
    CUDA_CHECK(cudaSetDevice(h->device));
    h->upload_f(level, f);
  });
}
// this rank's row block [begin, end) of amgb_hierarchy_local_range only (whole vector when the
// level is not sharded): no collective, 1/world of the host<->device bytes
int amgb_hierarchy_get_soln_local(amgb_hierarchy* h, int level, double* u_block) {
  return guarded([&] {
    if (!h || !u_block) throw std::invalid_argument("null argument");
    h->check_level(level);
    CUDA_CHECK(cudaSetDevice(h->device));
    h->download_local(level, true, u_block);
  });
}
int amgb_hierarchy_get_rhs_local(amgb_hierarchy* h, int level, double* f_block) {
  return guarded([&] {
    if (!h || !f_block) throw std::invalid_argument("null argument");
    h->check_level(level);
    CUDA_CHECK(cudaSetDevice(h->device));
    h->download_local(level, false, f_block);
  });
}
int amgb_hierarchy_set_soln_local(amgb_hierarchy* h, int level, const double* u_block) {
  return guarded([&] {
    if (!h || !u_block) throw std::invalid_argument("null argument");
    h->check_level(level);
    CUDA_CHECK(cudaSetDevice(h->device));
    h->upload_local(level, true, u_block);
  });
}
int amgb_hierarchy_set_rhs_local(amgb_hierarchy* h, int level, const double* f_block) {
  return guarded([&] {
    if (!h || !f_block) throw std::invalid_argument("null argument");
    h->check_level(level);
    CUDA_CHECK(cudaSetDevice(h->device));
    h->upload_local(level, false, f_block);
  });
}
int amgb_hierarchy_get_coloring(const amgb_hierarchy* h, int level, int* n_colors, int* color) {
  return guarded([&] {
    if (!h) throw std::invalid_argument("null argument");
    h->check_level(level);
    const Operator& A = *h->ops[level];
    if (!A.have_colors) throw ApiError(AMGB_ESTATE, "level has no colouring (smoother is not COLOR_GS)");
    if (n_colors) *n_colors = A.n_colors;
    if (color) std::memcpy(color, A.color.data(), sizeof(int) * A.color.size());
  });
}

int amgb_vcycle(amgb_hierarchy* h) {
  return guarded([&] {
    if (!h) throw std::invalid_argument("null argument");
    CUDA_CHECK(cudaSetDevice(h->device));
    h->vcycle();
  });
}
int amgb_vcycles(amgb_hierarchy* h, int64_t count) {
  return guarded([&] {
    if (!h) throw std::invalid_argument("null argument");
    CUDA_CHECK(cudaSetDevice(h->device));
    for (int64_t i = 0; i < count; ++i) h->vcycle();
    CUDA_CHECK(cudaStreamSynchronize(h->stream));
    h->check_halo();
  });
}
int amgb_hierarchy_rss(amgb_hierarchy* h, double* out) {
  return guarded([&] {
    if (!h || !out) throw std::invalid_argument("null argument");
    CUDA_CHECK(cudaSetDevice(h->device));
    *out = h->rss();
  });
}
int amgb_solve(amgb_hierarchy* h, int64_t* iters_done, double* last_error) {
  return guarded([&] {
    if (!h) throw std::invalid_argument("null argument");
    CUDA_CHECK(cudaSetDevice(h->device));
    // multigrid.hpp:311-337
    int64_t iter = 0;
    double error = 100;
    h->history.clear();
    const int64_t every = h->opt.compute_error_every_n_iters;
    while (iter < h->opt.n_iters && error > h->opt.tolerance) {
      h->vcycle();
      iter += 1;
      if (every != 0 && (iter % every) == 0) {
        error = h->rss();
        h->history.push_back(error);
      }
    }
    CUDA_CHECK(cudaStreamSynchronize(h->stream));
    h->check_halo();
    h->iters_done = iter;
    if (iters_done) *iters_done = iter;
    if (last_error) *last_error = error;
  });
}
int amgb_solve_relative(amgb_hierarchy* h, double rel_tol, int64_t* iters_done, double* last_rel) {
  return guarded([&] {
    if (!h) throw std::invalid_argument("null argument");
    CUDA_CHECK(cudaSetDevice(h->device));
    const double bnorm2 = h->rhs_sumsq();
    int64_t iter = 0;
    double rel = INFINITY;
    h->history.clear();
    const int64_t every = std::max<int64_t>(1, h->opt.compute_error_every_n_iters);
    while (iter < h->opt.n_iters && rel > rel_tol) {
      h->vcycle();
      iter += 1;
      if ((iter % every) == 0) {
        rel = std::sqrt(h->rss() / bnorm2);
        h->history.push_back(rel);
      }
    }
    CUDA_CHECK(cudaStreamSynchronize(h->stream));
    h->check_halo();
    h->iters_done = iter;
    if (iters_done) *iters_done = iter;
    if (last_rel) *last_rel = rel;
  });
}
// Conjugate gradients on A u = b preconditioned by one V-cycle from a zero guess (z = V(r)).
// The signs of a negative definite A (the reference's Laplacian, grid.hpp:62) cancel in
// alpha = (r.z) / (p.Ap) and beta, so the plain recurrences apply.  Needs a symmetric cycle
// (damped Jacobi or multicolour GS with equal pre- and post-smoothing, symmetric GS).
int amgb_solve_pcg(amgb_hierarchy* h, double rel_tol, int64_t max_iters, int64_t* iters_done,
                   double* last_rel_residual) {
  return guarded([&] {
    if (!h) throw std::invalid_argument("null argument");
    if (h->lv[0].sharded) throw ApiError(AMGB_ESTATE, "amgb_solve_pcg runs on a single GPU");
    CUDA_CHECK(cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    LevelState& S = h->lv[0];
    const int N = (int)h->n[0];
    const size_t bytes = sizeof(double) * (size_t)N;
    const int nb = std::max(1, blocks_for(N, 256));
    DevBuf<double> b, x, r, p, q, zero;
    for (DevBuf<double>* v : {&b, &x, &r, &p, &q, &zero}) v->alloc((size_t)N + 8);
    zero.zero(s);
    CUDA_CHECK(cudaMemcpyAsync(b.p, S.f.p, bytes, cudaMemcpyDeviceToDevice, s));
    CUDA_CHECK(cudaMemcpyAsync(x.p, S.u.p, bytes, cudaMemcpyDeviceToDevice, s));
    auto dot = [&](const double* a_, const double* b_) {
      LAUNCH(dev::k_dot_partial, nb, 256, 0, s, a_, b_, N, h->partial.p);
      LAUNCH(dev::k_sum_partials, 1, 256, 0, s, h->partial.p, nb, h->scalar.p);
      return h->finish_scalar_local();
    };
    h->ops[0]->residual(x.p, b.p, r.p, s);  // r = b - A x
    const double bnorm2 = dot(b.p, b.p);
    double rr = dot(r.p, r.p);
    double rel = bnorm2 > 0.0 ? std::sqrt(rr / bnorm2) : 0.0;
    h->history.clear();
    int64_t iter = 0;
    double rz_old = 0.0;
    while (iter < max_iters && rel > rel_tol) {
      // z = V(r): one cycle on A z = r from z = 0
      CUDA_CHECK(cudaMemcpyAsync(S.f.p, r.p, bytes, cudaMemcpyDeviceToDevice, s));
      CUDA_CHECK(cudaMemsetAsync(S.u.p, 0, bytes, s));
      h->vcycle();
      const double* z = S.u.p;
      const double rz = dot(r.p, z);
      if (iter == 0) CUDA_CHECK(cudaMemcpyAsync(p.p, z, bytes, cudaMemcpyDeviceToDevice, s));
      else LAUNCH(dev::k_xpay, nb, 256, 0, s, p.p, z, rz / rz_old, N);
      h->ops[0]->residual(p.p, zero.p, q.p, s);  // q = 0 - A p
      const double pq = dot(p.p, q.p);           // = -(p . A p)
      if (pq == 0.0 || !std::isfinite(pq)) break;
      const double alpha = -rz / pq;
      LAUNCH(dev::k_axpy, nb, 256, 0, s, x.p, alpha, p.p, N);
      LAUNCH(dev::k_axpy, nb, 256, 0, s, r.p, alpha, q.p, N);  // r -= alpha A p
      rz_old = rz;
      rr = dot(r.p, r.p);
      rel = std::sqrt(rr / bnorm2);
      h->history.push_back(rel);
      iter += 1;
    }
    CUDA_CHECK(cudaMemcpyAsync(S.f.p, b.p, bytes, cudaMemcpyDeviceToDevice, s));
    CUDA_CHECK(cudaMemcpyAsync(S.u.p, x.p, bytes, cudaMemcpyDeviceToDevice, s));
    CUDA_CHECK(cudaStreamSynchronize(s));
    h->iters_done = iter;
    if (iters_done) *iters_done = iter;
    if (last_rel_residual) *last_rel_residual = rel;
  });
}
// Restarted GMRES(m) on A x = b right-preconditioned by one V-cycle from a zero guess (M(v)), so the
// monitored quantity is the true residual.  Arnoldi with classical Gram-Schmidt and one
// reorthogonalisation on the device (krylov.cuh); the Hessenberg column, its Givens rotations and the
// back substitution on the host.  Specification: include/amgb.h, tests/oracle_gmres.py.
int amgb_solve_gmres(amgb_hierarchy* h, double rel_tol, int restart, int64_t max_iters, int64_t* iters_done,
                     double* last_rel_residual) {
  return guarded([&] {
    if (!h) throw std::invalid_argument("null argument");
    if (!(rel_tol >= 0.0)) throw std::invalid_argument("amgb_solve_gmres: rel_tol must be >= 0");
    if (restart < 1) throw std::invalid_argument("amgb_solve_gmres: restart must be >= 1");
    if (max_iters < 0) throw std::invalid_argument("amgb_solve_gmres: max_iters must be >= 0");
    if (h->lv[0].sharded) throw ApiError(AMGB_ESTATE, "amgb_solve_gmres runs on a single GPU");
    CUDA_CHECK(cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    LevelState& S = h->lv[0];
    const int64_t N = h->n[0];
    const size_t bytes = sizeof(double) * (size_t)N;
    const int m = restart;
    const int64_t ld = krylov::basis_ld(N);
    const int nb = krylov::tiles(N), nbv = std::max(1, blocks_for(N, krylov::kThreads));
    DevBuf<double> b, x, zero;
    for (DevBuf<double>* v : {&b, &x, &zero}) v->alloc((size_t)N + 8);
    zero.zero(s);
    CUDA_CHECK(cudaMemcpyAsync(b.p, S.f.p, bytes, cudaMemcpyDeviceToDevice, s));
    CUDA_CHECK(cudaMemcpyAsync(x.p, S.u.p, bytes, cudaMemcpyDeviceToDevice, s));
    auto sumsq = [&](const double* v) {
      LAUNCH(dev::k_sumsq_partial, nbv, 256, 0, s, v, (int)N, h->partial.p);
      LAUNCH(dev::k_sum_partials, 1, 256, 0, s, h->partial.p, nbv, h->scalar.p);
      return h->finish_scalar_local();
    };
    const double bnorm = std::sqrt(sumsq(b.p));
    h->history.clear();
    int64_t it = 0;
    double rel = 0.0;
    if (bnorm > 0.0) {
      // the (m + 1) x ld basis, the k x nb dot partials and one Hessenberg column (h, h', |w|^2)
      DevBuf<double> V, part, col;
      {
        const double want = (double)(m + 1) * (double)ld * sizeof(double);
        cudaError_t e = want < 9.0e18 ? cudaMalloc(&V.p, (size_t)(m + 1) * (size_t)ld * sizeof(double))
                                      : cudaErrorMemoryAllocation;
        if (e != cudaSuccess) {
          cudaGetLastError();
          V.p = nullptr;
          throw ApiError(AMGB_ECUDA, "amgb_solve_gmres: cannot allocate the Krylov basis of " +
                                         std::to_string(m + 1) + " x " + std::to_string(N) + " doubles (" +
                                         std::to_string(want / 1e9) + " GB): " + cudaGetErrorString(e));
        }
        V.n = (size_t)(m + 1) * (size_t)ld;
      }
      part.alloc((size_t)m * nb);
      col.alloc(2 * (size_t)m + 1);
      auto vec = [&](int i) { return V.p + (size_t)i * ld; };
      std::vector<double> H((size_t)(m + 1) * m), cs(m), sn(m), g(m + 1), y(m), hcol(2 * (size_t)m + 1);
      auto Hij = [&](int i, int j) -> double& { return H[(size_t)j * (m + 1) + i]; };
      // r = b - A x into v_0; the true relative residual
      auto true_residual = [&]() {
        h->ops[0]->residual(x.p, b.p, vec(0), s);
        return std::sqrt(sumsq(vec(0)));
      };
      double beta = true_residual();
      rel = beta / bnorm;
      bool failed = false;
      while (!failed && it < max_iters && rel > rel_tol) {
        LAUNCH(krylov::k_scale, nbv, krylov::kThreads, 0, s, vec(0), vec(0), beta, N);
        std::fill(g.begin(), g.end(), 0.0);
        g[0] = beta;
        int k = 0;  // Arnoldi steps of this cycle
        for (int j = 0; j < m && it < max_iters; ++j) {
          // w = A M(v_j) into v_{j+1}: a cycle on -v_j, then 0 - A z
          LAUNCH(krylov::k_negate, nbv, krylov::kThreads, 0, s, S.f.p, vec(j), N);
          CUDA_CHECK(cudaMemsetAsync(S.u.p, 0, bytes, s));
          h->vcycle();
          double* w = vec(j + 1);
          h->ops[0]->residual(S.u.p, zero.p, w, s);
          const int kk = j + 1;
          LAUNCH(krylov::k_multidot, nb, krylov::kThreads, 0, s, V.p, ld, kk, w, N, part.p);
          LAUNCH(krylov::k_sum_rows, kk, krylov::kThreads, 0, s, part.p, nb, col.p);
          LAUNCH(krylov::k_update<krylov::kDots>, nb, krylov::kThreads, 0, s, w, w, V.p, ld, kk, col.p, N, part.p);
          LAUNCH(krylov::k_sum_rows, kk, krylov::kThreads, 0, s, part.p, nb, col.p + kk);
          LAUNCH(krylov::k_update<krylov::kSumSq>, nb, krylov::kThreads, 0, s, w, w, V.p, ld, kk, col.p + kk, N,
                 part.p);
          LAUNCH(krylov::k_sum_rows, 1, krylov::kThreads, 0, s, part.p, nb, col.p + 2 * kk);
          CUDA_CHECK(cudaMemcpyAsync(hcol.data(), col.p, sizeof(double) * (2 * kk + 1), cudaMemcpyDeviceToHost, s));
          CUDA_CHECK(cudaStreamSynchronize(s));
          bool finite = true;
          for (int i = 0; i < kk; ++i) {
            Hij(i, j) = hcol[i] + hcol[kk + i];
            finite = finite && std::isfinite(Hij(i, j));
          }
          const double hnext = std::sqrt(hcol[2 * kk]);
          Hij(j + 1, j) = hnext;
          if (!finite || !std::isfinite(hnext)) {  // abandon the cycle: x stays that of the last one
            failed = true;
            break;
          }
          if (hnext != 0.0) LAUNCH(krylov::k_scale, nbv, krylov::kThreads, 0, s, w, w, hnext, N);
          for (int i = 0; i < j; ++i) {
            const double t = cs[i] * Hij(i, j) + sn[i] * Hij(i + 1, j);
            Hij(i + 1, j) = -sn[i] * Hij(i, j) + cs[i] * Hij(i + 1, j);
            Hij(i, j) = t;
          }
          const double d = std::hypot(Hij(j, j), hnext);
          if (d == 0.0) {  // A M v_j = 0: singular, no rotation
            failed = true;
            break;
          }
          cs[j] = Hij(j, j) / d;
          sn[j] = hnext / d;
          Hij(j, j) = d;
          Hij(j + 1, j) = 0.0;
          g[j + 1] = -sn[j] * g[j];
          g[j] = cs[j] * g[j];
          k = j + 1;
          it += 1;
          const double est = std::fabs(g[j + 1]) / bnorm;
          h->history.push_back(est);
          if (est <= rel_tol || hnext == 0.0) break;
        }
        if (failed || k == 0) break;
        // y = H(0:k, 0:k) \ g(0:k); t = V_k y (c = -y from a zero base) into f_0; x += M(t)
        for (int i = k - 1; i >= 0; --i) {
          double acc = g[i];
          for (int q = i + 1; q < k; ++q) acc -= Hij(i, q) * y[q];
          y[i] = acc / Hij(i, i);
        }
        for (int i = 0; i < k; ++i) hcol[i] = -y[i];
        CUDA_CHECK(cudaMemcpyAsync(col.p, hcol.data(), sizeof(double) * k, cudaMemcpyHostToDevice, s));
        LAUNCH(krylov::k_update<krylov::kNone>, nb, krylov::kThreads, 0, s, S.f.p, nullptr, V.p, ld, k, col.p, N,
               nullptr);
        CUDA_CHECK(cudaMemsetAsync(S.u.p, 0, bytes, s));
        h->vcycle();
        LAUNCH(dev::k_axpy, nbv, 256, 0, s, x.p, 1.0, S.u.p, (int)N);
        beta = true_residual();
        rel = beta / bnorm;
      }
    }
    CUDA_CHECK(cudaMemcpyAsync(S.f.p, b.p, bytes, cudaMemcpyDeviceToDevice, s));
    CUDA_CHECK(cudaMemcpyAsync(S.u.p, x.p, bytes, cudaMemcpyDeviceToDevice, s));
    CUDA_CHECK(cudaStreamSynchronize(s));
    h->iters_done = it;
    if (iters_done) *iters_done = it;
    if (last_rel_residual) *last_rel_residual = rel;
  });
}
int64_t amgb_hierarchy_iters_done(const amgb_hierarchy* h) { return h ? h->iters_done : 0; }
int64_t amgb_hierarchy_error_history(const amgb_hierarchy* h, double* out, int64_t cap) {
  if (!h) return 0;
  const int64_t nh = (int64_t)h->history.size();
  if (out) std::memcpy(out, h->history.data(), sizeof(double) * std::min(cap, nh));
  return nh;
}
int amgb_synchronize(amgb_hierarchy* h) {
  return guarded([&] {
    if (!h) throw std::invalid_argument("null argument");
    CUDA_CHECK(cudaStreamSynchronize(h->stream));
    h->check_halo();
  });
}

int amgb_restrict(amgb_hierarchy* h, int level, const double* r_fine, double* f_coarse) {
  return guarded([&] {
    if (!h || !r_fine || !f_coarse) throw std::invalid_argument("null argument");
    h->check_level(level, true);
    h->require_whole(level);
    CUDA_CHECK(cudaSetDevice(h->device));
    DevBuf<double> r, fc;
    r.upload(r_fine, h->n[level], h->stream);
    fc.alloc(h->n[level + 1]);
    if (h->sa())
      h->restrict_sa(r.p, fc.p, nullptr, level, h->stream);
    else if (h->bilinear())
      h->restrict2d(r.p, fc.p, level, h->stream);
    else
      LAUNCH(dev::k_restrict, blocks_for(h->n[level + 1], 256), 256, 0, h->stream, r.p, (int)h->n[level],
             fc.p, (int)h->n[level + 1]);
    fc.download(f_coarse, h->stream);
    CUDA_CHECK(cudaStreamSynchronize(h->stream));
  });
}
int amgb_prolong_add(amgb_hierarchy* h, int level, const double* e_coarse, double* u_fine) {
  return guarded([&] {
    if (!h || !e_coarse || !u_fine) throw std::invalid_argument("null argument");
    h->check_level(level, true);
    h->require_whole(level);
    CUDA_CHECK(cudaSetDevice(h->device));
    DevBuf<double> e, uf;
    e.upload(e_coarse, h->n[level + 1], h->stream);
    uf.upload(u_fine, h->n[level], h->stream);
    if (h->sa())
      h->prolong_add_sa(e.p, uf.p, level, h->stream);
    else if (h->bilinear())
      h->prolong_add2d(e.p, uf.p, level, h->stream);
    else
      LAUNCH(dev::k_prolong_add, blocks_for(h->n[level], 256), 256, 0, h->stream, e.p, 0, (int)h->n[level + 1],
             uf.p, 0, (int)h->n[level]);
    uf.download(u_fine, h->stream);
    CUDA_CHECK(cudaStreamSynchronize(h->stream));
  });
}
int amgb_smooth_level(amgb_hierarchy* h, int level) {
  return guarded([&] {
    if (!h) throw std::invalid_argument("null argument");
    h->check_level(level);
    CUDA_CHECK(cudaSetDevice(h->device));
    h->prepare_smoother(level);
    h->smooth(level, h->stream);
    CUDA_CHECK(cudaStreamSynchronize(h->stream));
  });
}
int amgb_residual_level(amgb_hierarchy* h, int level, double* r) {
  return guarded([&] {
    if (!h || !r) throw std::invalid_argument("null argument");
    h->check_level(level);
    h->require_whole(level);
    CUDA_CHECK(cudaSetDevice(h->device));
    DevBuf<double> rd;
    rd.alloc(h->n[level]);
    h->ops[level]->residual(h->lv[level].u.p, h->lv[level].f.p, rd.p, h->stream);
    rd.download(r, h->stream);
    CUDA_CHECK(cudaStreamSynchronize(h->stream));
  });
}
int amgb_residual_restrict_level(amgb_hierarchy* h, int level) {
  return guarded([&] {
    if (!h) throw std::invalid_argument("null argument");
    h->check_level(level, true);
    CUDA_CHECK(cudaSetDevice(h->device));
    h->residual_restrict(level, h->stream);
    CUDA_CHECK(cudaStreamSynchronize(h->stream));
  });
}
int amgb_coarse_solve(amgb_hierarchy* h) {
  return guarded([&] {
    if (!h) throw std::invalid_argument("null argument");
    CUDA_CHECK(cudaSetDevice(h->device));
    h->coarse_solve(h->stream);
    CUDA_CHECK(cudaStreamSynchronize(h->stream));
  });
}

int amgb_hierarchy_tail_first(const amgb_hierarchy* h) { return h ? h->tail_first : -1; }
int amgb_hierarchy_mid_range(const amgb_hierarchy* h, int* first, int* end, int* tile_rows, int* blocks) {
  if (!h) return AMGB_EINVAL;
  if (first) *first = h->mid_first;
  if (end) *end = h->mid_end;
  if (tile_rows) *tile_rows = h->mid_first >= 0 ? h->midp.T : 0;
  if (blocks) *blocks = h->mid_first >= 0 ? h->midp.n_blocks : 0;
  return AMGB_OK;
}
int amgb_hierarchy_fused_legs(const amgb_hierarchy* h, int level) {
  return (h && h->leg_ok(level)) ? 1 : 0;
}
int amgb_hierarchy_matrix_free(const amgb_hierarchy* h, int level) {
  return (h && h->leg_ok(level) && h->legs[level].matrix_free) ? 1 : 0;
}
int amgb_hierarchy_dictionary_types(const amgb_hierarchy* h, int level) {
  return (h && h->leg_ok(level)) ? h->legs[level].dict_types : 0;
}
int amgb_hierarchy_leg_plan(const amgb_hierarchy* h, int level, int up, int64_t* info) {
  return guarded([&] {
    if (!h || !info) throw std::invalid_argument("null argument");
    h->check_level(level);
    if (!h->leg_ok(level)) throw ApiError(AMGB_ESTATE, "level has no fused legs");
    if (h->legs[level].stream) {
      const sleg::Params& P = up ? h->legs[level].sup : h->legs[level].sdown;
      info[0] = P.m;
      info[1] = 1;
      info[2] = P.Wu;
      info[3] = P.LJ;
      info[4] = (P.n_warps + 3) / 4;
      info[5] = P.n_strips;
      info[6] = 2;
      info[7] = 128;
      info[8] = 0;
      info[9] = (32 - P.Wu) / 2 - (up ? 0 : 1);
      return;
    }
    const leg::Plan& pl = up ? h->legs[level].up : h->legs[level].down;
    info[0] = pl.P.m;
    info[1] = pl.P.rho;
    info[2] = pl.P.W;
    info[3] = pl.P.LJ;
    info[4] = pl.tiles;
    info[5] = pl.P.n_strips;
    info[6] = pl.P.PF;
    info[7] = pl.threads;
    info[8] = (int64_t)pl.smem_bytes;
    info[9] = pl.P.NS;
  });
}

// Device-side Galerkin product of one level (SURVEY.md section 8f rank 1, not yet part of the
// setup): computes A_{level+1} = R (A_level P) from the level's device mirror with k_galerkin_dia,
// times it, and compares every diagonal bit for bit with the mirror of level + 1 that the host
// setup produced.  mismatches = number of differing entries (0 expected).
int amgb_hierarchy_galerkin_device(amgb_hierarchy* h, int level, double* ms_out, int64_t* mismatches) {
  return guarded([&] {
    if (!h) throw std::invalid_argument("null argument");
    h->check_level(level, true);
    h->require_whole(level);
    h->require_whole(level + 1);
    CUDA_CHECK(cudaSetDevice(h->device));
    const DevMat& F = h->ops[level]->rows_of_A();
    const DevMat& Cm = h->ops[level + 1]->rows_of_A();
    if (h->sa()) throw ApiError(AMGB_ESTATE, "the device-side Galerkin product covers the grid transfers only");
    if (!F.is_dia || !Cm.is_dia || F.dia.rows.p || Cm.dia.rows.p)
      throw ApiError(AMGB_ESTATE, "the device-side Galerkin product needs the DIA layout");
    gal::FineDia A;
    A.n = (int)h->n[level];
    A.nd = F.dia.n_diag;
    A.ld = F.dia.ld;
    for (int d = 0; d < A.nd; ++d) A.off[d] = F.dia.off[d];
    A.val = F.dia.val.p;
    CoarseOffsets oc{};
    const bool bl = h->bilinear();
    const int nd_c = bl ? gal::coarse_offsets_2d((int)h->m[level + 1], oc.v) : gal::coarse_offsets(A.nd, A.off, oc.v);
    if (nd_c < 0) throw ApiError(AMGB_ESTATE, "coarse operator has too many diagonals");
    const int n_c = (int)h->n[level + 1];
    const int ld_c = (n_c + 31) / 32 * 32;
    DevBuf<double> out;
    out.alloc((size_t)nd_c * ld_c);
    out.zero(h->stream);
    cudaEvent_t e0, e1;
    CUDA_CHECK(cudaEventCreate(&e0));
    CUDA_CHECK(cudaEventCreate(&e1));
    auto once = [&] {
      if (bl)
        LAUNCH(k_galerkin_dia2d, blocks_for(n_c, 256), 256, 0, h->stream, A, (int)h->m[level], (int)h->m[level + 1], nd_c,
               oc, out.p, ld_c);
      else
        LAUNCH(k_galerkin_dia, blocks_for(n_c, 256), 256, 0, h->stream, A, n_c, nd_c, oc, out.p, ld_c);
    };
    once();  // warm-up
    CUDA_CHECK(cudaEventRecord(e0, h->stream));
    once();
    CUDA_CHECK(cudaEventRecord(e1, h->stream));
    CUDA_CHECK(cudaEventSynchronize(e1));
    float ms = 0.f;
    CUDA_CHECK(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    if (ms_out) *ms_out = ms;
    // compare with the HOST Galerkin product of level + 1 (rows of A in DIA, built from the host
    // chain -- in device-setup mode that chain is rebuilt here on demand), diagonal by diagonal, and
    // with the mirror of level + 1 the hierarchy actually uses
    const Csc& Mh = h->host_matrix(level + 1);
    Csc MhT = transpose(Mh);
    Dia want_d = build_dia(bitwise_equal(Mh, MhT) ? Mh : MhT);
    if (!want_d.ok) throw ApiError(AMGB_ESTATE, "host coarse operator does not fit the DIA layout");
    std::vector<double> got((size_t)nd_c * ld_c), used((size_t)Cm.dia.n_diag * Cm.dia.ld);
    CUDA_CHECK(cudaMemcpy(got.data(), out.p, got.size() * sizeof(double), cudaMemcpyDeviceToHost));
    CUDA_CHECK(cudaMemcpy(used.data(), Cm.dia.val.p, used.size() * sizeof(double), cudaMemcpyDeviceToHost));
    int64_t bad = 0;
    std::vector<char> matched(nd_c, 0);
    for (int d = 0; d < want_d.n_diag; ++d) {
      int c = -1, u = -1;
      for (int k = 0; k < nd_c; ++k)
        if (oc.v[k] == want_d.off[d]) c = k;
      for (int k = 0; k < Cm.dia.n_diag; ++k)
        if (Cm.dia.off[k] == want_d.off[d]) u = k;
      if (c < 0 || u < 0) {
        bad += n_c;
        continue;
      }
      matched[c] = 1;
      for (int i = 0; i < n_c; ++i) {
        const double w = want_d.val[(size_t)d * want_d.ld + i];
        bad += std::memcmp(&got[(size_t)c * ld_c + i], &w, 8) != 0;
        bad += std::memcmp(&used[(size_t)u * Cm.dia.ld + i], &w, 8) != 0;
      }
    }
    if (Cm.dia.n_diag != want_d.n_diag) bad += n_c;
    for (int c = 0; c < nd_c; ++c)  // diagonals the host operator does not have must be all zero
      if (!matched[c])
        for (int i = 0; i < n_c; ++i) bad += (got[(size_t)c * ld_c + i] != 0.0);
    if (mismatches) *mismatches = bad;
  });
}

// Mean milliseconds of the four phases of a V-cycle on this rank over `reps` un-captured cycles:
// out[0] sharded down legs, out[1] gather of the first replicated right-hand side, out[2] the levels
// below the sharded ones (both directions; on one GPU: everything), out[3] sharded up legs.
// Collective on a sharded hierarchy (every rank runs the same cycles).
int amgb_hierarchy_phase_times(amgb_hierarchy* h, int reps, double* out) {
  return guarded([&] {
    if (!h || !out || reps < 1) throw std::invalid_argument("bad argument");
    CUDA_CHECK(cudaSetDevice(h->device));
    cudaEvent_t ev[5];
    for (auto& e : ev) CUDA_CHECK(cudaEventCreate(&e));
    for (int k = 0; k < 4; ++k) out[k] = 0.0;
    for (int i = 0; i < reps + 1; ++i) {
      h->phase_ev = ev;
      try {
        h->enqueue_vcycle(h->stream);
      } catch (...) {
        h->phase_ev = nullptr;
        throw;
      }
      h->phase_ev = nullptr;
      CUDA_CHECK(cudaStreamSynchronize(h->stream));
      if (i == 0) continue;  // warm-up
      for (int k = 0; k < 4; ++k) {
        float ms = 0.f;
        CUDA_CHECK(cudaEventElapsedTime(&ms, ev[k], ev[k + 1]));
        out[k] += ms / reps;
      }
    }
    for (auto& e : ev) cudaEventDestroy(e);
    h->check_halo();
  });
}

int64_t amgb_kernel_launches(void) { return g_launches.load(); }
int64_t amgb_hierarchy_launches_per_vcycle(const amgb_hierarchy* h) {
  return h ? h->launches_per_vcycle : 0;
}
int64_t amgb_hierarchy_pass_bytes(const amgb_hierarchy* h, int level) {
  if (!h || level < 0 || level >= h->L) return -1;
  return 12 * h->ops[level]->nnz_device() + 28 * h->n[level] + 4;
}
int64_t amgb_hierarchy_vcycle_bytes(const amgb_hierarchy* h) {
  // SURVEY.md section 8d: per non-coarsest level 4 smoother passes + 1 residual
  // (= 5 B_l) + restriction/prolongation vectors (24 N_l + 16 N_{l+1}); scaled by
  // the smoother passes actually configured.
  if (!h) return -1;
  int64_t total = 0;
  const int64_t passes_per_smooth =
      h->opt.smoother == AMGB_SMOOTHER_JACOBI ? h->opt.smoother_iters : 2 * h->opt.smoother_iters;
  for (int l = 0; l + 1 < h->L; ++l) {
    const int64_t B = amgb_hierarchy_pass_bytes(h, l);
    total += (2 * passes_per_smooth + 1) * B;
    if (h->sa())  // k_restrict_sa and k_prolong_add_sa stream R and P (12 B per entry each) besides the vectors
      total += 12 * (h->sa_R_rows[l].nnz + h->sa_P_rows[l].nnz) + 24 * h->n[l] + 24 * h->n[l + 1];
    else
      total += 24 * h->n[l] + 16 * h->n[l + 1];
  }
  return total;
}

int amgb_hierarchy_format(const amgb_hierarchy* h, int level) {
  if (!h || level < 0 || level >= h->L) return -1;
  return h->ops[level]->rows_of_A().is_dia ? AMGB_FORMAT_DIA : AMGB_FORMAT_SELL;
}
// diagonals a fused leg streams from the level's DIA mirror (0 for SELL), 8 bytes per row each: all of
// them, or the centre and upper ones on a half-streamed level
int amgb_hierarchy_n_diagonals(const amgb_hierarchy* h, int level) {
  if (!h || level < 0 || level >= h->L) return -1;
  const DevMat& A = h->ops[level]->rows_of_A();
  if (!A.is_dia) return 0;
  if (h->leg_ok(level) && h->legs[level].stream && h->legs[level].half) return A.dia.n_diag / 2 + 1;
  return A.dia.n_diag;
}
int amgb_hierarchy_gs_kernel(const amgb_hierarchy* h, int level) {
  if (!h || level < 0 || level >= h->L || h->opt.smoother != AMGB_SMOOTHER_GS) return -1;
  const Operator& A = *h->ops[level];  // the schedules were built when the hierarchy was created
  if (h->opt.gs_mode == AMGB_GS_AUTO && A.wave_ok) return AMGB_GS_KERNEL_WAVE;
  if ((h->opt.gs_mode == AMGB_GS_AUTO || h->opt.gs_mode == AMGB_GS_LINESCAN) && A.lines_ok) return AMGB_GS_KERNEL_LINESCAN;
  return AMGB_GS_KERNEL_FRONTS;
}
int64_t amgb_hierarchy_matrix_bytes(const amgb_hierarchy* h, int level) {
  if (!h || level < 0 || level >= h->L) return -1;
  return h->ops[level]->rows_of_A().stored_bytes();
}

int amgb_time_kernel(amgb_hierarchy* h, int level, int kind, int warmup, int reps, double* ms_out) {
  return guarded([&] {
    if (!h || !ms_out || reps < 1) throw std::invalid_argument("bad argument");
    if (kind == 9 || kind == 11) {
      // 9: one damped-Jacobi sweep, 11: one residual of `level`, on a sharded level INCLUDING the halo
      // exchange with ranks +-1 (SURVEY.md 8d config 4: the smoother + residual microbenchmark).
      // Collective on a sharded hierarchy.  The level's iterate is restored afterwards.
      h->check_level(level);
      CUDA_CHECK(cudaSetDevice(h->device));
      cudaStream_t s = h->stream;
      LevelState& S = h->lv[level];
      if (!S.tmp.p) S.tmp.alloc(S.n_vec() + 8);
      DevBuf<double> keep;
      keep.alloc(S.u.n);
      CUDA_CHECK(cudaMemcpyAsync(keep.p, S.u.p, sizeof(double) * S.u.n, cudaMemcpyDeviceToDevice, s));
      double* src = S.u.p;
      double* dst = S.tmp.p;
      auto once = [&] {
        h->site_cursor = amgb_hierarchy::kMaxSites - 1;  // reserved site of out-of-cycle exchanges
        if (kind == 9) {
          h->jacobi_sweep(level, src, dst, s);
          std::swap(src, dst);
        } else {
          h->exchange(level, S.u.p, s);
          h->ops[level]->residual(S.u_own(), S.f.p, S.tmp_own(), s);
        }
      };
      for (int i = 0; i < warmup; ++i) once();
      cudaEvent_t e0, e1;
      CUDA_CHECK(cudaEventCreate(&e0));
      CUDA_CHECK(cudaEventCreate(&e1));
      CUDA_CHECK(cudaEventRecord(e0, s));
      for (int i = 0; i < reps; ++i) once();
      CUDA_CHECK(cudaEventRecord(e1, s));
      CUDA_CHECK(cudaEventSynchronize(e1));
      float ms = 0.f;
      CUDA_CHECK(cudaEventElapsedTime(&ms, e0, e1));
      cudaEventDestroy(e0);
      cudaEventDestroy(e1);
      CUDA_CHECK(cudaMemcpyAsync(S.u.p, keep.p, sizeof(double) * S.u.n, cudaMemcpyDeviceToDevice, s));
      CUDA_CHECK(cudaStreamSynchronize(s));
      h->site_cursor = 0;
      h->check_halo();
      *ms_out = (double)ms / reps;
      return;
    }
    if (kind >= 6 && kind <= 8) {
      // 6 / 7: the mid-level down / up kernel, 8: the coarse tail (or the coarsest solve alone).  They are
      // timed on the live level state (a cycle's worth of it): nothing to restore, every run computes
      // the same values from the same inputs.
      CUDA_CHECK(cudaSetDevice(h->device));
      cudaStream_t s = h->stream;
      if ((kind == 6 || kind == 7) && h->mid_first < 0) throw ApiError(AMGB_ESTATE, "no mid levels");
      auto once = [&] {
        if (kind == 6) h->mid_down(s);
        else if (kind == 7) h->mid_up(s);
        else if (h->tail_first > 0) h->launch_tail(s);
        else h->coarse_solve(s);
      };
      for (int i = 0; i < warmup; ++i) once();
      cudaEvent_t e0, e1;
      CUDA_CHECK(cudaEventCreate(&e0));
      CUDA_CHECK(cudaEventCreate(&e1));
      CUDA_CHECK(cudaEventRecord(e0, s));
      for (int i = 0; i < reps; ++i) once();
      CUDA_CHECK(cudaEventRecord(e1, s));
      CUDA_CHECK(cudaEventSynchronize(e1));
      float ms = 0.f;
      CUDA_CHECK(cudaEventElapsedTime(&ms, e0, e1));
      cudaEventDestroy(e0);
      cudaEventDestroy(e1);
      *ms_out = (double)ms / reps;
      return;
    }
    h->check_level(level, kind == 2 || kind == 3);
    if (kind == 2 || kind == 3) h->require_whole(level);
    if ((kind == 12 || kind == 13) && h->opt.smoother != AMGB_SMOOTHER_LINE_GS)
      throw ApiError(AMGB_ESTATE, "kinds 12 and 13 time the passes of a line Gauss-Seidel hierarchy");
    if (kind == 4 || kind == 5) {
      // fused down / up leg of this level; they work on the level state, which is restored
      if (!h->leg_ok(level)) throw ApiError(AMGB_ESTATE, "level has no fused legs");
      CUDA_CHECK(cudaSetDevice(h->device));
      cudaStream_t s = h->stream;
      LevelState& S = h->lv[level];
      LevelState& C = h->lv[level + 1];
      DevBuf<double> su, sf;
      su.alloc(S.u.n);
      sf.alloc(C.f.n);
      CUDA_CHECK(cudaMemcpyAsync(su.p, S.u.p, sizeof(double) * S.u.n, cudaMemcpyDeviceToDevice, s));
      CUDA_CHECK(cudaMemcpyAsync(sf.p, C.f.p, sizeof(double) * C.f.n, cudaMemcpyDeviceToDevice, s));
      auto once = [&] {
        if (kind == 4) h->leg_down(level, s);
        else h->leg_up(level, s);
      };
      for (int i = 0; i < warmup; ++i) once();
      cudaEvent_t e0, e1;
      CUDA_CHECK(cudaEventCreate(&e0));
      CUDA_CHECK(cudaEventCreate(&e1));
      CUDA_CHECK(cudaEventRecord(e0, s));
      for (int i = 0; i < reps; ++i) once();
      CUDA_CHECK(cudaEventRecord(e1, s));
      CUDA_CHECK(cudaEventSynchronize(e1));
      float ms = 0.f;
      CUDA_CHECK(cudaEventElapsedTime(&ms, e0, e1));
      cudaEventDestroy(e0);
      cudaEventDestroy(e1);
      CUDA_CHECK(cudaMemcpyAsync(S.u.p, su.p, sizeof(double) * S.u.n, cudaMemcpyDeviceToDevice, s));
      CUDA_CHECK(cudaMemcpyAsync(C.f.p, sf.p, sizeof(double) * C.f.n, cudaMemcpyDeviceToDevice, s));
      CUDA_CHECK(cudaStreamSynchronize(s));
      *ms_out = (double)ms / reps;
      return;
    }
    CUDA_CHECK(cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    h->prepare_smoother(level);
    Operator& A = *h->ops[level];
    LevelState& S = h->lv[level];
    if (!S.tmp.p) S.tmp.alloc(S.n_vec() + 4);
    if (kind == 12 || kind == 13)  // the other direction's factors are built on first use
      A.ensure_line_gs((int)h->m[level], kind == 12 ? lgs::kX : lgs::kY, h->fast_arith(),
                       "level " + std::to_string(level), s);
    DevBuf<double> scratch_u, scratch_c, scratch_c2;
    scratch_u.alloc(S.n_vec());
    CUDA_CHECK(cudaMemcpyAsync(scratch_u.p, S.u.p, sizeof(double) * S.n_vec(), cudaMemcpyDeviceToDevice, s));
    double* su = scratch_u.p + S.halo_lo;  // first owned row (no halo exchange is timed here)
    if (kind == 2 || kind == 3) {
      scratch_c.alloc(h->n[level + 1]);
      scratch_c.zero(s);
      scratch_c2.alloc(h->n[level + 1]);
    }
    auto once = [&] {
      switch (kind) {
        case 0:
          if (h->opt.smoother == AMGB_SMOOTHER_JACOBI)
            A.jacobi(su, S.f.p, h->opt.omega, S.tmp_own(), s);
          else if (h->opt.smoother == AMGB_SMOOTHER_COLOR_GS)
            for (int c = 0; c < A.n_colors; ++c) A.color_pass(c, S.f.p, scratch_u.p, s);
          else if (h->opt.smoother == AMGB_SMOOTHER_LINE_GS)
            A.line_gs_half(true, h->opt.lines, h->fast_arith(), S.f.p, scratch_u.p, S.tmp.p, s);
          else
            A.gs_direction(true, S.f.p, scratch_u.p, S.tmp.p, h->opt.gs_mode, s);
          break;
        case 1:
          A.residual(su, S.f.p, S.tmp_own(), s);
          break;
        case 2:
          if (h->sa())  // the restriction alone: its residual is a separate k_residual launch (kind 1)
            h->restrict_sa(scratch_u.p, scratch_c2.p, scratch_c.p, level, s);
          else if (h->bilinear())
            A.residual_restrict2d(scratch_u.p, S.f.p, (int)h->m[level], 0, scratch_c2.p, scratch_c.p, (int)h->m[level + 1],
                                  0, 0, (int)h->m[level + 1], s);
          else
            A.residual_restrict(scratch_u.p, S.f.p, scratch_c2.p, scratch_c.p, (int)h->n[level + 1], s);
          break;
        case 3:
          if (h->sa())
            h->prolong_add_sa(scratch_c.p, scratch_u.p, level, s);
          else if (h->bilinear())
            h->prolong_add2d(scratch_c.p, scratch_u.p, level, s);
          else
            LAUNCH(dev::k_prolong_add2, blocks_for((h->n[level] + 1) / 2, 256), 256, 0, s, scratch_c.p, 0,
                   (int)h->n[level + 1], scratch_u.p, 0, (int)h->n[level]);
          break;
        case 12:
        case 13:
          A.line_pass(kind == 12 ? lgs::kX : lgs::kY, 0, h->fast_arith(), S.f.p, scratch_u.p, S.tmp.p, s);
          break;
        default:
          throw std::invalid_argument("unknown kernel kind");
      }
    };
    for (int i = 0; i < warmup; ++i) once();
    cudaEvent_t e0, e1;
    CUDA_CHECK(cudaEventCreate(&e0));
    CUDA_CHECK(cudaEventCreate(&e1));
    CUDA_CHECK(cudaEventRecord(e0, s));
    for (int i = 0; i < reps; ++i) once();
    CUDA_CHECK(cudaEventRecord(e1, s));
    CUDA_CHECK(cudaEventSynchronize(e1));
    float ms = 0.f;
    CUDA_CHECK(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    *ms_out = (double)ms / reps;
  });
}

}  // extern "C"
