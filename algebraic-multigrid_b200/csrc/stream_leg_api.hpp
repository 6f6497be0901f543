// Parameters and host-side dispatch of the register-streaming fused V-cycle legs
// (kernels: stream_leg.cuh, compiled in legs.cu).
#pragma once
#include <cstdint>

#include <cuda_runtime.h>

namespace amgb {
namespace sleg {

enum Kind { DOWN_U = 0, DOWN_ZERO = 1, UP = 2 };

// stencil slot sl = (a + 1) * 3 + (delta + 1), ascending in column order
constexpr unsigned kMask5 = 0x0BAu;   // (-1,0) (0,-1) (0,0) (0,1) (1,0): level 0 of an n x n grid, m = n
constexpr unsigned kMask7a = 0x1BBu;  // level 1 with m = its smaller far offset: (-1,-1) (-1,0) (0,*) (1,0) (1,1)
constexpr unsigned kMask7b = 0x0FEu;  // level 1 with m = its larger far offset:  (-1,0) (-1,1) (0,*) (1,-1) (1,0)
constexpr unsigned kMask9 = 0x1FFu;   // Galerkin levels >= 2

// Fused halo push of a row-block sharded level (multi-GPU): the rows of an output vector that a
// neighbouring rank keeps as ghost rows are stored straight into that rank's copy of the vector
// (peer-mapped pointer, the stores travel over NVLink) by the warps that produced them.
struct Push {
  double* dst;  // neighbour's vector, shifted so that dst[i] is the neighbour's element for my local index i
  int begin;    // my local indices [begin, end) go to the neighbour (empty: begin >= end)
  int end;
};

// Per-launch synchronisation with the two neighbouring ranks.  Every leg kernel of the sharded
// cycle is a "site"; all ranks run the same sequence of sites.  side 0 = lower neighbour (rank
// g-1), side 1 = upper neighbour.  The warps whose chunk lies next to a block edge ("edge warps")
//   * first wait until the neighbour on that side has finished ITS edge warps of the previous
//     site: its pushes into my ghost rows have landed (read-after-write) and it has stopped
//     reading the ghost rows I am about to overwrite (write-after-read);
//   * at the end push their boundary rows, fence, and count themselves done; the last one bumps
//     this site's epoch and releases it into the neighbour's flag.
// Epochs and counters live in device memory, so a replayed CUDA graph keeps counting.
struct Sync {
  int enabled;                          // 0: single GPU, nothing below is touched
  int edge_lo_chunks;                   // chunks [0, edge_lo_chunks) are lower-edge chunks
  int edge_hi_chunk0;                   // chunks [edge_hi_chunk0, n_chunks) are upper-edge chunks
  int expected[2];                      // edge warps per side
  const unsigned long long* wait_flag[2];   // my flag the neighbour raised at the previous site (nullptr: no neighbour)
  const unsigned long long* wait_epoch[2];  // my own epoch of the previous site = the value to wait for
  unsigned long long* epoch[2];         // this site's epoch counters
  unsigned long long* peer_flag[2];     // the neighbour's flag for this site (nullptr: no neighbour)
  unsigned int* done[2];                // this site's edge-warp counters (self-resetting)
  int* timed_out;                       // set when a wait gives up (mapped host memory)
  long long timeout_cycles;
  Push push_u[2];                       // uout rows -> neighbours
  Push push_fc[2];                      // fc entries (local coarse indices) -> neighbours
};

struct Params {
  // The kernel works on a WINDOW of the level: local row k is global row base + k.  A whole level
  // is the window [0, n) with base 0; a rank of the row-block sharded cycle passes its block plus
  // the ghost rows on both sides (which the neighbours' previous kernels have filled) and stores
  // results for its own rows only -- the ghost rows are recomputed redundantly, like the lanes at
  // a warp's edge.
  int base;       // global row of local row 0 (may be negative: rows before the level start)
  int n_global;   // rows of the level
  int own_begin;  // local rows [own_begin, own_end) are stored
  int own_end;
  int cbase;      // global coarse index of fc[0] and e[0]
  int n_e;        // entries of e / fc that exist locally
  int nu;         // Jacobi sweeps per smooth call (selects the kernel instantiation on the host)
  int n;         // rows of the window
  int m;         // line length
  int n_lines;   // ceil(n / m)
  int Wu;        // owned elements per warp (32 - 2H)
  int n_strips;  // ceil(m / Wu)
  int LJ;        // lines per chunk
  int LJ_edge;   // lines of the FIRST and the LAST chunk (= LJ on one GPU; half of it on a sharded level, so
                 // that the warps which wait for / push to a neighbour have less streaming to do and the
                 // flag latency hides behind the other chunks)
  int n_chunks;
  int n_warps;   // n_strips * n_chunks
  int ld;
  int n_coarse;
  // derived by finish() below
  int row_lo, row_hi1;  // local rows that exist: [row_lo, row_hi1] = window ∩ level (loads are clamped to it)
  int e_lo, e_cnt;      // local coarse indices that exist: [e_lo, e_lo + e_cnt)
  int l2_ahead;         // > 0: prefetch the line this many steps beyond the register ring into L2
  // matrix-free five-point variant (the operator was VERIFIED to be cst[] on the five offsets -m, -1,
  // 0, +1, +m wherever the neighbour exists and empty elsewhere): no operator row is loaded
  int matrix_free;
  double cst[5];
  // row-type dictionary variant (the operator has at most 256 distinct rows, VERIFIED at setup): one
  // byte per row selects a row of the table, which every block copies into shared memory
  int dict_types;              // 0: off
  const unsigned char* tid;    // type of every row of the window
  const double* table;         // dict_types x (number of diagonals)
  // half streaming (the operator was VERIFIED to be bitwise symmetric): only vd[] of the centre and
  // upper diagonals are read, the lower coefficients come from registers
  int half;
  double omega;
  const double* val;
  const double* vd[9];  // val + d * ld
  const double* f;
  const double* uin;
  const double* e;
  double* uout;
  double* fc;
  Sync sync;

  // first line and number of lines of chunk c
  __host__ __device__ int chunk_begin(int c) const { return c == 0 ? 0 : LJ_edge + (c - 1) * LJ; }
  __host__ __device__ int chunk_lines(int c) const { return (c == 0 || c == n_chunks - 1) ? LJ_edge : LJ; }
  // chunk geometry for `chunks` chunks over n_lines lines; edge_half: the two edge chunks get half the lines
  void set_chunks(int chunks, bool edge_half) {
    if (chunks < 1) chunks = 1;
    if (!edge_half || chunks < 4) {
      LJ = (n_lines + chunks - 1) / chunks;
      LJ_edge = LJ;
      n_chunks = (n_lines + LJ - 1) / LJ;
    } else {
      LJ = (n_lines + chunks - 2) / (chunks - 1);  // two half chunks + (chunks - 2) whole ones
      LJ_edge = (LJ + 1) / 2;
      n_chunks = 2;
      while (2 * LJ_edge + (n_chunks - 2) * LJ < n_lines) ++n_chunks;
    }
    n_warps = n_strips * n_chunks;
  }
  // fills the derived fields; call after every other field is set
  void finish(int n_diag) {
    for (int d = 0; d < 9; ++d) vd[d] = val + (size_t)(d < n_diag ? d : 0) * (size_t)ld;
    row_lo = base < 0 ? -base : 0;
    const int hi = (n < n_global - base) ? n : n_global - base;
    row_hi1 = hi - 1 > row_lo ? hi - 1 : row_lo;
    e_lo = cbase < 0 ? -cbase : 0;
    const int ehi = (n_e < n_coarse - cbase) ? n_e : n_coarse - cbase;
    e_cnt = ehi > e_lo ? ehi - e_lo : 0;
  }
};

// Which chunks are "edge chunks" of a sharded leg (host): those that read ghost rows -- their stages
// reach NS + 1 lines beyond the chunk -- or that produce rows / coarse entries a neighbour receives.
// lo_reach / hi_reach: local fine rows below / from which every producer must be an edge chunk
// (own_begin / own_end widened by the push ranges).  Fills edge_lo_chunks, edge_hi_chunk0, expected[].
inline void classify_edges(const Params& P, int NS, int lo_reach, int hi_reach, Sync& Y) {
  const long long lo_bound = (long long)lo_reach + (long long)(NS + 2) * P.m;
  const long long hi_bound = (long long)hi_reach - (long long)(NS + 2) * P.m;
  Y.edge_lo_chunks = 0;  // chunks whose first row lies below lo_bound
  while (Y.edge_lo_chunks < P.n_chunks && (long long)P.chunk_begin(Y.edge_lo_chunks) * P.m < lo_bound) ++Y.edge_lo_chunks;
  if (Y.edge_lo_chunks < 1) Y.edge_lo_chunks = 1;
  Y.edge_hi_chunk0 = P.n_chunks - 1;  // first chunk whose last row lies above hi_bound
  while (Y.edge_hi_chunk0 > 0 &&
         (long long)(P.chunk_begin(Y.edge_hi_chunk0 - 1) + P.chunk_lines(Y.edge_hi_chunk0 - 1)) * P.m > hi_bound)
    --Y.edge_hi_chunk0;
  Y.expected[0] = Y.edge_lo_chunks * P.n_strips;
  Y.expected[1] = (P.n_chunks - Y.edge_hi_chunk0) * P.n_strips;
}

__host__ __device__ constexpr int popc9(unsigned v) {
  int c = 0;
  for (int i = 0; i < 9; ++i) c += (v >> i) & 1u;
  return c;
}
// slot mask mirrored through the centre (slot sl -> 8 - sl: offset o -> -o)
__host__ __device__ constexpr unsigned mirror9(unsigned v) {
  unsigned r = 0;
  for (int i = 0; i < 9; ++i) r |= ((v >> i) & 1u) << (8 - i);
  return r;
}
// lanes lost on each side of a warp: one per chained stencil stage (+ 1 for the restriction)
__host__ __device__ constexpr int stages(int kind, int nu) { return kind == DOWN_U ? nu + 1 : nu; }
__host__ __device__ constexpr int lost_lanes(int kind, int nu) { return stages(kind, nu) + (kind == UP ? 0 : 1); }

// Host-side dispatch (legs.cu).  action 0: does a kernel exist for (kind, mask, nu)?  1: launch on
// `s` (returns true when a kernel was launched).  2: set the L1 carve-out (outside stream capture)
// and report the resident warps per SM the register count allows in *warps_per_sm.
// fast: AMGB_ARITH_FAST kernels (FMA + refined reciprocal) instead of the reference-order ones.
// Params::matrix_free selects the matrix-free five-point kernels (kMask5 only), Params::half the
// half-streaming ones.
bool dispatch(int kind, unsigned mask, const Params& P, cudaStream_t s, int action, int* warps_per_sm, bool fast);

}  // namespace sleg
}  // namespace amgb
