// Host-side (cold) setup for the B200 V-cycle path: CSC container, the
// reference's interpolation operators and Galerkin coarse operators, greedy
// colouring, banded LDL^T of the coarsest operator, Gauss-Seidel dependency
// schedules and the SELL-32 device layout.  Pure C++17, no CUDA, no Eigen.
//
// Reference behaviour restated here (paths relative to the reference root):
//   include/amg/interpolator.hpp:106-141  LinearInterpolator::make_operators
//   include/amg/multigrid.hpp:127-130     n_H_dofs_from_n_h_dofs
//   include/amg/multigrid.hpp:211-237     hierarchy loop, A_H = R*(A*P)
//   include/amg/multigrid.hpp:240-243     coarsest factorisation
//   include/amg/grid.hpp:31-140           problem generators
#pragma once
#include <cstdint>
#include <string>
#include <vector>

namespace amgb {

struct Csc {
  int rows = 0, cols = 0;
  std::vector<int> colptr;  // cols + 1
  std::vector<int> rowidx;  // ascending inside each column
  std::vector<double> val;
  int64_t nnz() const { return colptr.empty() ? 0 : colptr.back(); }
  int64_t nnz_nonzero() const;
};

Csc csc_from_arrays(int rows, int cols, const int* colptr, const int* rowidx, const double* val);
Csc transpose(const Csc& A);
bool bitwise_equal(const Csc& A, const Csc& B);

// ---- generators (grid.hpp) ----
double grid_spacing_h(int64_t n);
Csc grid_laplacian(int64_t n, double eps_y);
void grid_rhs(int64_t n, double* b);

// ---- interpolation + Galerkin ----
int64_t coarse_dofs(int64_t fine_dofs);
Csc make_prolongation(int64_t n_h, int64_t n_H);
// Bilinear transfer on an m x m grid (DOF k = y*m + x): m_H = m_h / 2 lines per coarse level, so
// every fine line is covered by some coarse line also when m_h is even; P = P1 (x) P1 with P1 =
// make_prolongation(m_h, m_H), columns in ascending coarse index, rows ascending inside a column.
int64_t coarse_lines_2d(int64_t m_h);
Csc make_prolongation_2d(int64_t m_h, int64_t m_H);
// m with m * m == n, or -1
int64_t grid_lines(int64_t n);
// Smoothed aggregation (AMGB_TRANSFER_SMOOTHED_AGGREGATION, specification in include/amgb.h and
// tests/oracle_sa.py).  Row i of A is CSC column i.  sa_aggregate fills agg (one aggregate id per row,
// ids in creation order) and returns the number of aggregates; sa_prolongation returns the smoothed P
// (A.cols x n_agg).  Both throw std::invalid_argument naming `level` (and the row) on a zero diagonal;
// sa_aggregate also on a strength threshold below 0 or NaN.
int64_t sa_aggregate(const Csc& A, double theta, std::vector<int>& agg, int level = 0);
// The two steps of sa_aggregate, so that the device setup (setup_sa.cuh builds the strength graph) runs the
// same passes: sa_strength fills the strong-neighbour lists (CSR, ascending; same checks as sa_aggregate),
// sa_aggregate_passes runs passes 1-3 on them.
void sa_strength(const Csc& A, double theta, std::vector<int>& sptr, std::vector<int>& snb, int level = 0);
int64_t sa_aggregate_passes(int n, const int* sptr, const int* snb, std::vector<int>& agg);
// the std::invalid_argument messages of a zero diagonal and of a level 0 that does not reduce
std::string sa_zero_diagonal_message(int level, int row);
std::string sa_no_reduction_message(int rows, int64_t n_agg);
Csc sa_prolongation(const Csc& A, const std::vector<int>& agg, int64_t n_agg, int level = 0);
// The levels: mats[0] = A, then P[l] and mats[l + 1] = R (A P) with R = P^T while l + 1 < n_levels and
// level l has more than kSaMaxCoarse rows.  A coarse level whose aggregation does not reduce it ends the
// hierarchy as its coarsest level; when level 0 does not reduce, std::invalid_argument.  phase_s, when
// given, accumulates the seconds spent in [aggregation, prolongators, Galerkin products].
constexpr int kSaMaxCoarse = 200;
void sa_hierarchy(Csc&& A, double theta, int n_levels, std::vector<Csc>& mats, std::vector<Csc>& P,
                  double* phase_s = nullptr);
// Eigen 3.4.0 conservative ColMajor product: entry (i,j) = sum over ascending k
// of L(i,k)*R(k,j); numerical zeros kept; result columns sorted.
Csc multiply(const Csc& L, const Csc& R);
Csc galerkin(const Csc& R, const Csc& A, const Csc& P);

// ---- greedy first-fit colouring of the (pruned, symmetrised) graph ----
int greedy_coloring(const Csc& A, const Csc& AT, std::vector<int>& color);

// ---- coarsest level: banded LDL^T, natural order, no pivoting ----
struct BandedLdlt {
  int n = 0, bw = 0;
  std::vector<double> L;  // n * max(bw,1): L[i*bw + (j-(i-bw))] = L(i,j), i-bw <= j < i
  std::vector<double> d;  // n
};
BandedLdlt factor_banded_ldlt(const Csc& A);

// ---- SELL-32 layout of "row c = CSC column c", explicit zeros dropped ----
// Slice s holds rows [32 s, 32 s + 32) of `rows` (or of 0..n-1 when rows is
// empty); element j of lane t sits at slice_ptr[s] + 32 j + t.  Padding has
// col = -1.  Entries keep their ascending column order, so a thread that walks
// j = 0.. reproduces the reference's summation order.
struct Sell {
  int n_rows = 0;    // rows covered (== rows.size() when a subset)
  int n_slices = 0;
  int64_t nnz = 0;   // real entries
  std::vector<uint32_t> slice_ptr;  // n_slices + 1
  std::vector<int> col;
  std::vector<double> val;
  std::vector<int> rows;  // optional row subset (ascending), empty = identity
};
Sell build_sell(const Csc& M, const std::vector<int>* rows = nullptr);

// ---- DIA layout (diagonal storage) of "row c = CSC column c" ----
// For the banded operators of this path (5/7/9 distinct offsets per level) the
// column index of entry d of row r is r + off[d], so no index array is
// streamed and the x gathers do not depend on a prior load.  val[d*ld + t] is
// the entry of the t-th covered row on diagonal d (0.0 = absent; explicit
// zeros are dropped exactly like in the SELL layout).  off is ascending, so
// walking d = 0.. keeps the reference's ascending-column summation order.
struct Dia {
  bool ok = false;   // false: too many distinct offsets, use SELL
  int n_rows = 0;
  int n_cols = 0;
  int ld = 0;        // n_rows rounded up to 32
  int n_diag = 0;
  int64_t nnz = 0;   // real entries
  std::vector<int> off;
  std::vector<double> val;  // n_diag * ld
  std::vector<int> rows;    // optional row subset
  // bit d of mask[s] set <=> diagonal d has an entry among rows [32 s, 32 s + 32); filled only
  // when skipping empty slices saves at least a tenth of the matrix bytes, else empty
  std::vector<unsigned short> mask;
};
constexpr int kMaxDiag = 16;
Dia build_dia(const Csc& M, const std::vector<int>* rows = nullptr);
// Rows [row_begin, row_begin + n_rows) of M with local numbering: entry d of
// local row t multiplies x_local[t + off[d] + x_shift], x_local being this
// rank's halo-extended vector (x_shift = number of halo elements below).
Dia build_dia_block(const Csc& M, int row_begin, int n_rows);
// Same for a window that may reach past the ends of the matrix (those rows stay empty), with the
// diagonal order given by `offsets` (ascending); !ok when an entry falls outside them.
Dia build_dia_window(const Csc& M, int row_begin, int n_rows, const std::vector<int>& offsets);

// ---- row-block partition of the fine levels over the ranks of one node ----
// Level l < n_sharded is split into contiguous row blocks [start[l][g], start[l][g+1]);
// block starts at level 0 are multiples of 2^n_sharded so that the coarse block of
// a rank is exactly the image of its fine block (coarse row J belongs to the owner of
// fine row 2J+1).  halo_lo / halo_hi are the u-halo widths a rank keeps below / above
// its block (half-bandwidth w_l, plus `ghost` on the upper side); `ghost` is the number
// of extra rows [end, end+ghost) whose residual the rank forms itself so that the fused
// residual+restriction needs no second exchange: ghost_l = 2*ghost_{l+1} + 1.
struct PartitionPlan {
  int world = 1;
  int n_levels = 0;
  int n_sharded = 0;                        // levels [0, n_sharded) are sharded
  std::vector<int64_t> n;                   // level sizes
  std::vector<std::vector<int64_t>> start;  // [level][rank 0..world]
  std::vector<int> halo_lo, halo_hi, ghost; // per sharded level
};
// max_sharded caps the number of sharded levels (the rest is agglomerated).
PartitionPlan make_partition_plan(const std::vector<int64_t>& level_sizes,
                                  const std::vector<int>& half_bandwidth, int world,
                                  int64_t min_rows_per_rank, int max_sharded = 1 << 30);
// Plan of a bilinear 2-D hierarchy (m_l x m_l grids, m_{l+1} = m_l / 2): blocks of whole grid lines.
// Level 0 gets the line starts Y0(g) = floor(m_0 g / world) rounded down to a multiple of 2^n_sharded,
// level l the lines Y0(g) >> l (the last rank ends at m_l); start = line * m_l, so a coarse block
// starts exactly at half its fine block's first line.  Coarse line J restricts fine lines 2J..2J+2,
// hence ghost lines ghost_{ns-1} = 1, ghost_l = 2 ghost_{l+1} + 1; in rows ghost = lines * m_l,
// halo_lo = m_l + 2 (the +-(m_l + 1) stencil plus a margin) and halo_hi = (ghost lines + 1) m_l + 2.
// Level l is sharded while m_l^2 / world >= min_rows_per_rank (never the coarsest level), and
// n_sharded shrinks until every block holds at least max(halo_lo, halo_hi) rows.
PartitionPlan make_partition_plan_2d(const std::vector<int64_t>& lines_per_level, int world,
                                     int64_t min_rows_per_rank);

// ---- Gauss-Seidel wavefront schedule on the pruned dependency DAG ----
// forward: row k depends on rows j<k with M(j,k) != 0 (column k of M used as
// row k); backward: rows j>k.  order lists rows grouped by wavefront.
struct Schedule {
  std::vector<int> order;      // n
  std::vector<int> front_ptr;  // n_fronts + 1
  int n_fronts() const { return (int)front_ptr.size() - 1; }
  int max_width = 0;
};
Schedule gs_schedule(const Csc& M, bool forward);

}  // namespace amgb
