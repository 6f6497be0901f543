// See host_setup.hpp.  Everything here runs once per hierarchy (cold path).
#include "host_setup.hpp"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstring>
#include <limits>
#include <stdexcept>

namespace amgb {

int64_t Csc::nnz_nonzero() const {
  int64_t c = 0;
  for (double v : val) c += (v != 0.0);
  return c;
}

Csc csc_from_arrays(int rows, int cols, const int* colptr, const int* rowidx, const double* val) {
  Csc A;
  A.rows = rows;
  A.cols = cols;
  A.colptr.assign(colptr, colptr + cols + 1);
  const int64_t nnz = colptr[cols];
  A.rowidx.assign(rowidx, rowidx + nnz);
  A.val.assign(val, val + nnz);
  return A;
}

Csc transpose(const Csc& A) {
  Csc T;
  T.rows = A.cols;
  T.cols = A.rows;
  const int64_t nnz = A.nnz();
  T.colptr.assign((size_t)A.rows + 1, 0);
  T.rowidx.resize(nnz);
  T.val.resize(nnz);
  for (int64_t p = 0; p < nnz; ++p) T.colptr[A.rowidx[p] + 1]++;
  for (int r = 0; r < A.rows; ++r) T.colptr[r + 1] += T.colptr[r];
  std::vector<int> cursor(T.colptr.begin(), T.colptr.end() - 1);
  for (int c = 0; c < A.cols; ++c)
    for (int p = A.colptr[c]; p < A.colptr[c + 1]; ++p) {
      const int q = cursor[A.rowidx[p]]++;
      T.rowidx[q] = c;  // ascending because c ascends
      T.val[q] = A.val[p];
    }
  return T;
}

bool bitwise_equal(const Csc& A, const Csc& B) {
  if (A.rows != B.rows || A.cols != B.cols || A.colptr != B.colptr || A.rowidx != B.rowidx)
    return false;
  return A.val.size() == B.val.size() &&
         std::memcmp(A.val.data(), B.val.data(), A.val.size() * sizeof(double)) == 0;
}

// ------------------------------------------------------------------ generators

double grid_spacing_h(int64_t n) { return 2.0 / static_cast<double>(n + 1); }  // grid.hpp:31

// grid.hpp:50-98: D = tridiag(1,-2,1)/(h*h); A = kron(I,D) + eps_y*kron(D,I).
// With DOF k = line*n + pos the first term couples k+-1 inside a line and the
// second couples k+-n; eps_y == 1 is the reference operator.
Csc grid_laplacian(int64_t n, double eps_y) {
  const double hh = grid_spacing_h(n) * grid_spacing_h(n);
  const double d_off = 1.0 / hh, d_dia = -2.0 / hh;
  const double line_off = d_off, cross_off = eps_y * d_off;
  const double dia = d_dia + eps_y * d_dia;
  const int64_t N = n * n;
  Csc A;
  A.rows = A.cols = static_cast<int>(N);
  A.colptr.resize(N + 1);
  A.rowidx.reserve(5 * N - 4 * n);
  A.val.reserve(5 * N - 4 * n);
  for (int64_t k = 0; k < N; ++k) {
    const int64_t line = k / n, pos = k % n;
    A.colptr[k] = static_cast<int>(A.rowidx.size());
    auto put = [&](int64_t r, double v) {
      A.rowidx.push_back(static_cast<int>(r));
      A.val.push_back(v);
    };
    if (line > 0) put(k - n, cross_off);
    if (pos > 0) put(k - 1, line_off);
    put(k, dia);
    if (pos + 1 < n) put(k + 1, line_off);
    if (line + 1 < n) put(k + n, cross_off);
  }
  A.colptr[N] = static_cast<int>(A.rowidx.size());
  return A;
}

// grid.hpp:108-140: interior points of LinSpaced(n+2,-1,1); x_i = -1 + i*step
// (Eigen's linspaced_op: low + i*step, no fused multiply-add); line index is
// the outer loop and the first argument of f.
void grid_rhs(int64_t n, double* b) {
  const double step = 2.0 / static_cast<double>(n + 1);
  std::vector<double> x(n + 2);
  for (int64_t i = 0; i < n + 2; ++i) x[i] = -1.0 + static_cast<double>(i) * step;
  x[n + 1] = 1.0;
  for (int64_t line = 1; line <= n; ++line) {
    const double xl = x[line];
    double* out = b + (line - 1) * n;
    for (int64_t pos = 1; pos <= n; ++pos) {
      const double xp = x[pos];
      out[pos - 1] = 5 * std::exp(-10 * (xl * xl + xp * xp));
    }
  }
}

// ------------------------------------------------------- interpolation/Galerkin

int64_t coarse_dofs(int64_t fine_dofs) {  // multigrid.hpp:127-130 (size_t arithmetic)
  return static_cast<int64_t>((static_cast<uint64_t>(fine_dofs) + 1) / 2 - 1);
}

// interpolator.hpp:106-130: column j of P = {(2j, .5), (2j+1, 1), (2j+2, .5)},
// each kept only when the row is inside [0, n_h).
Csc make_prolongation(int64_t n_h, int64_t n_H) {
  Csc P;
  P.rows = static_cast<int>(n_h);
  P.cols = static_cast<int>(n_H);
  P.colptr.resize(n_H + 1);
  P.rowidx.reserve(3 * n_H);
  P.val.reserve(3 * n_H);
  static const double w[3] = {0.5, 1.0, 0.5};
  for (int64_t j = 0; j < n_H; ++j) {
    P.colptr[j] = static_cast<int>(P.rowidx.size());
    for (int t = 0; t < 3; ++t) {
      const int64_t r = 2 * j + t;
      if (r < n_h) {
        P.rowidx.push_back(static_cast<int>(r));
        P.val.push_back(w[t]);
      }
    }
  }
  P.colptr[n_H] = static_cast<int>(P.rowidx.size());
  return P;
}

int64_t coarse_lines_2d(int64_t m_h) { return m_h / 2; }

Csc make_prolongation_2d(int64_t m_h, int64_t m_H) {
  const Csc P1 = make_prolongation(m_h, m_H);
  const int64_t rows = m_h * m_h, cols = m_H * m_H;
  if (rows > std::numeric_limits<int>::max() || 9 * cols > std::numeric_limits<int>::max())
    throw std::overflow_error("make_prolongation_2d: exceeds int32 indexing");
  Csc P;
  P.rows = static_cast<int>(rows);
  P.cols = static_cast<int>(cols);
  P.colptr.resize(cols + 1);
  P.rowidx.reserve(9 * cols);
  P.val.reserve(9 * cols);
  // column (Y, X): rows (y, x) for y in column Y of P1, x in column X of P1, y-major = ascending row
  for (int64_t Y = 0; Y < m_H; ++Y)
    for (int64_t X = 0; X < m_H; ++X) {
      P.colptr[Y * m_H + X] = static_cast<int>(P.rowidx.size());
      for (int p = P1.colptr[Y]; p < P1.colptr[Y + 1]; ++p)
        for (int q = P1.colptr[X]; q < P1.colptr[X + 1]; ++q) {
          P.rowidx.push_back(static_cast<int>(P1.rowidx[p] * m_h + P1.rowidx[q]));
          P.val.push_back(P1.val[p] * P1.val[q]);
        }
    }
  P.colptr[cols] = static_cast<int>(P.rowidx.size());
  return P;
}

int64_t grid_lines(int64_t n) {
  if (n < 0) return -1;
  int64_t m = static_cast<int64_t>(std::llround(std::sqrt(static_cast<double>(n))));
  while (m > 0 && m * m > n) --m;
  while ((m + 1) * (m + 1) <= n) ++m;
  return m * m == n ? m : -1;
}

// ------------------------------------------------------- smoothed aggregation

std::string sa_zero_diagonal_message(int level, int row) {
  return "smoothed aggregation: level " + std::to_string(level) + " has a zero diagonal at row " + std::to_string(row);
}

std::string sa_no_reduction_message(int rows, int64_t n_agg) {
  return "smoothed aggregation: the aggregation of level 0 does not reduce it (" + std::to_string(rows) + " rows, " +
         std::to_string(n_agg) + " aggregates)";
}

// a_ii of every row (row i = CSC column i); a zero or absent diagonal is rejected
static std::vector<double> sa_diagonal(const Csc& A, int level) {
  std::vector<double> d(A.cols, 0.0);
  for (int i = 0; i < A.cols; ++i)
    for (int p = A.colptr[i]; p < A.colptr[i + 1]; ++p)
      if (A.rowidx[p] == i) d[i] = A.val[p];
  for (int i = 0; i < A.cols; ++i)
    if (d[i] == 0.0) throw std::invalid_argument(sa_zero_diagonal_message(level, i));
  return d;
}

void sa_strength(const Csc& A, double theta, std::vector<int>& sptr, std::vector<int>& snb, int level) {
  if (!(theta >= 0.0))
    throw std::invalid_argument("smoothed aggregation: strength must be >= 0, got " + std::to_string(theta));
  if (A.rows != A.cols) throw std::invalid_argument("smoothed aggregation: A must be square");
  const int n = A.cols;
  const std::vector<double> d = sa_diagonal(A, level);
  // strong neighbours of row i, ascending: |a_ij| > theta * sqrt(|a_ii| * |a_jj|), j != i, a_ij != 0
  sptr.assign((size_t)n + 1, 0);
  snb.clear();
  snb.reserve(A.nnz());
  for (int i = 0; i < n; ++i) {
    for (int p = A.colptr[i]; p < A.colptr[i + 1]; ++p) {
      const int j = A.rowidx[p];
      const double a = A.val[p];
      if (j == i || a == 0.0) continue;
      const double thr = theta * std::sqrt(std::fabs(d[i]) * std::fabs(d[j]));
      if (std::fabs(a) > thr) snb.push_back(j);
    }
    sptr[i + 1] = static_cast<int>(snb.size());
  }
}

int64_t sa_aggregate_passes(int n, const int* sptr, const int* snb, std::vector<int>& agg) {
  agg.assign(n, -1);
  int64_t count = 0;
  for (int i = 0; i < n; ++i) {  // pass 1: i and all its strong neighbours free -> new aggregate
    if (agg[i] >= 0) continue;
    bool free_nbrs = true;
    for (int p = sptr[i]; p < sptr[i + 1] && free_nbrs; ++p) free_nbrs = agg[snb[p]] < 0;
    if (!free_nbrs) continue;
    const int J = static_cast<int>(count++);
    agg[i] = J;
    for (int p = sptr[i]; p < sptr[i + 1]; ++p) agg[snb[p]] = J;
  }
  const std::vector<int> pass1 = agg;
  for (int i = 0; i < n; ++i) {  // pass 2: join the pass-1 aggregate of the first such strong neighbour
    if (agg[i] >= 0) continue;
    for (int p = sptr[i]; p < sptr[i + 1]; ++p)
      if (pass1[snb[p]] >= 0) {
        agg[i] = pass1[snb[p]];
        break;
      }
  }
  for (int i = 0; i < n; ++i) {  // pass 3: new aggregate with the still free strong neighbours
    if (agg[i] >= 0) continue;
    const int J = static_cast<int>(count++);
    agg[i] = J;
    for (int p = sptr[i]; p < sptr[i + 1]; ++p)
      if (agg[snb[p]] < 0) agg[snb[p]] = J;
  }
  return count;
}

int64_t sa_aggregate(const Csc& A, double theta, std::vector<int>& agg, int level) {
  std::vector<int> sptr, snb;
  sa_strength(A, theta, sptr, snb, level);
  return sa_aggregate_passes(A.cols, sptr.data(), snb.data(), agg);
}

Csc sa_prolongation(const Csc& A, const std::vector<int>& agg, int64_t n_agg, int level) {
  const int n = A.cols;
  const std::vector<double> d = sa_diagonal(A, level);
  // Gershgorin bound of D^-1 A over the stored entries
  double rho = 0.0;
  for (int i = 0; i < n; ++i) {
    double s = 0.0;
    for (int p = A.colptr[i]; p < A.colptr[i + 1]; ++p) s += std::fabs(A.val[p]);
    rho = std::max(rho, s / std::fabs(d[i]));
  }
  const double w = (4.0 / 3.0) / rho;
  // rows of P, built as the CSC columns of R = P^T
  Csc R;
  R.rows = static_cast<int>(n_agg);
  R.cols = n;
  R.colptr.assign((size_t)n + 1, 0);
  std::vector<int> slot(n_agg, -1), touched;
  std::vector<double> sums;
  for (int i = 0; i < n; ++i) {
    touched.clear();
    sums.clear();
    for (int p = A.colptr[i]; p < A.colptr[i + 1]; ++p) {
      const int J = agg[A.rowidx[p]];
      if (slot[J] < 0) {
        slot[J] = static_cast<int>(touched.size());
        touched.push_back(J);
        sums.push_back(0.0);
      }
      sums[slot[J]] += A.val[p];
    }
    const double c = w / d[i];
    std::vector<int> order(touched.size());
    for (size_t t = 0; t < order.size(); ++t) order[t] = static_cast<int>(t);
    std::sort(order.begin(), order.end(), [&](int a, int b) { return touched[a] < touched[b]; });
    for (int t : order) {
      const int J = touched[t];
      const double prod = c * sums[t];
      R.rowidx.push_back(J);
      R.val.push_back((J == agg[i] ? 1.0 : 0.0) - prod);
    }
    for (int J : touched) slot[J] = -1;
    if (R.rowidx.size() > static_cast<size_t>(std::numeric_limits<int>::max()))
      throw std::overflow_error("sa_prolongation: P exceeds int32 indexing");
    R.colptr[i + 1] = static_cast<int>(R.rowidx.size());
  }
  return transpose(R);
}

void sa_hierarchy(Csc&& A, double theta, int n_levels, std::vector<Csc>& mats, std::vector<Csc>& P,
                  double* phase_s) {
  using clock = std::chrono::steady_clock;
  auto lap = [&](clock::time_point& t0, int phase) {
    const clock::time_point t1 = clock::now();
    if (phase_s) phase_s[phase] += std::chrono::duration<double>(t1 - t0).count();
    t0 = t1;
  };
  mats.clear();
  P.clear();
  mats.push_back(std::move(A));
  while (static_cast<int>(mats.size()) < n_levels && mats.back().cols > kSaMaxCoarse) {
    const int l = static_cast<int>(mats.size()) - 1;
    std::vector<int> agg;
    clock::time_point t0 = clock::now();
    const int64_t n_agg = sa_aggregate(mats[l], theta, agg, l);
    lap(t0, 0);
    if (n_agg >= mats[l].cols) {
      // level 0 (a diagonal matrix, say) has no hierarchy at all; a coarse level whose couplings are all weak
      // (the Galerkin levels turn dense a few hundred rows above the 200-row target on large problems)
      // becomes the coarsest level
      if (l == 0) throw std::invalid_argument(sa_no_reduction_message(mats[l].cols, n_agg));
      break;
    }
    P.push_back(sa_prolongation(mats[l], agg, n_agg, l));
    lap(t0, 1);
    Csc AH = galerkin(transpose(P.back()), mats[l], P.back());
    mats.push_back(std::move(AH));
    lap(t0, 2);
  }
}

Csc multiply(const Csc& L, const Csc& R) {
  if (L.cols != R.rows) throw std::invalid_argument("multiply: inner dimensions differ");
  Csc C;
  C.rows = L.rows;
  C.cols = R.cols;
  C.colptr.assign((size_t)R.cols + 1, 0);
  // sparse accumulator: slot[i] = position of row i in the current column, or -1
  std::vector<int> slot(L.rows, -1);
  std::vector<int> touched;
  std::vector<double> sums;
  std::vector<int> perm;
  C.rowidx.reserve(static_cast<size_t>(R.nnz()) * 2);
  C.val.reserve(static_cast<size_t>(R.nnz()) * 2);
  for (int j = 0; j < R.cols; ++j) {
    touched.clear();
    sums.clear();
    for (int q = R.colptr[j]; q < R.colptr[j + 1]; ++q) {
      const int k = R.rowidx[q];
      const double y = R.val[q];
      for (int p = L.colptr[k]; p < L.colptr[k + 1]; ++p) {
        const int i = L.rowidx[p];
        const double term = L.val[p] * y;
        if (slot[i] < 0) {
          slot[i] = static_cast<int>(touched.size());
          touched.push_back(i);
          sums.push_back(term);
        } else {
          sums[slot[i]] += term;
        }
      }
    }
    perm.resize(touched.size());
    for (size_t t = 0; t < perm.size(); ++t) perm[t] = static_cast<int>(t);
    std::sort(perm.begin(), perm.end(), [&](int a, int b) { return touched[a] < touched[b]; });
    for (int t : perm) {
      C.rowidx.push_back(touched[t]);
      C.val.push_back(sums[t]);
    }
    for (int i : touched) slot[i] = -1;
    if (C.rowidx.size() > static_cast<size_t>(std::numeric_limits<int>::max()))
      throw std::overflow_error("multiply: result exceeds int32 indexing");
    C.colptr[j + 1] = static_cast<int>(C.rowidx.size());
  }
  return C;
}

Csc galerkin(const Csc& R, const Csc& A, const Csc& P) {  // multigrid.hpp:219-223
  return multiply(R, multiply(A, P));
}

// ------------------------------------------------------------------ colouring

int greedy_coloring(const Csc& A, const Csc& AT, std::vector<int>& color) {
  const int N = A.cols;
  color.assign(N, -1);
  std::vector<int> stamp;  // stamp[c] == k  <=>  colour c is taken by a neighbour of k
  int n_colors = 0;
  for (int k = 0; k < N; ++k) {
    for (const Csc* M : {&A, &AT})
      for (int p = M->colptr[k]; p < M->colptr[k + 1]; ++p) {
        const int j = M->rowidx[p];
        if (j >= k || M->val[p] == 0.0) continue;
        stamp[color[j]] = k;  // color[j] < n_colors <= stamp.size()
      }
    int c = 0;
    while (c < n_colors && stamp[c] == k) ++c;
    color[k] = c;
    if (c == n_colors) {
      ++n_colors;
      stamp.push_back(-1);
    }
  }
  return n_colors;
}

// ------------------------------------------------------------------ banded LDLT

BandedLdlt factor_banded_ldlt(const Csc& A) {
  BandedLdlt F;
  const int n = A.cols;
  int bw = 0;
  for (int c = 0; c < n; ++c)
    for (int p = A.colptr[c]; p < A.colptr[c + 1]; ++p) bw = std::max(bw, A.rowidx[p] - c);
  F.n = n;
  F.bw = bw;
  const int ld = std::max(bw, 1);
  F.L.assign(static_cast<size_t>(n) * ld, 0.0);
  F.d.assign(n, 0.0);
  // lower band of A, row-major: band[i*(bw+1) + (j - (i-bw))]
  const int w = bw + 1;
  std::vector<double> band(static_cast<size_t>(n) * w, 0.0);
  for (int c = 0; c < n; ++c)
    for (int p = A.colptr[c]; p < A.colptr[c + 1]; ++p) {
      const int r = A.rowidx[p];
      if (r >= c) band[static_cast<size_t>(r) * w + (c - (r - bw))] = A.val[p];
    }
  auto Lij = [&](int i, int j) -> double& { return F.L[static_cast<size_t>(i) * ld + (j - (i - bw))]; };
  for (int i = 0; i < n; ++i) {
    const int first = std::max(0, i - bw);
    for (int j = first; j < i; ++j) {
      double s = band[static_cast<size_t>(i) * w + (j - (i - bw))];
      for (int k = std::max(first, j - bw); k < j; ++k) s -= Lij(i, k) * F.d[k] * Lij(j, k);
      Lij(i, j) = s / F.d[j];
    }
    double s = band[static_cast<size_t>(i) * w + bw];
    for (int k = first; k < i; ++k) s -= Lij(i, k) * F.d[k] * Lij(i, k);
    F.d[i] = s;
  }
  return F;
}

// ------------------------------------------------------------------ SELL-32

Sell build_sell(const Csc& M, const std::vector<int>* rows) {
  Sell S;
  const int n = rows ? static_cast<int>(rows->size()) : M.cols;
  S.n_rows = n;
  S.n_slices = (n + 31) / 32;
  S.slice_ptr.assign((size_t)S.n_slices + 1, 0);
  if (rows) S.rows = *rows;
  auto row_of = [&](int t) { return rows ? (*rows)[t] : t; };
  auto real_len = [&](int r) {
    int c = 0;
    for (int p = M.colptr[r]; p < M.colptr[r + 1]; ++p) c += (M.val[p] != 0.0);
    return c;
  };
  uint64_t total = 0;
  for (int s = 0; s < S.n_slices; ++s) {
    int width = 0;
    for (int t = 32 * s; t < std::min(n, 32 * s + 32); ++t) width = std::max(width, real_len(row_of(t)));
    S.slice_ptr[s] = static_cast<uint32_t>(total);
    total += 32ull * width;
    if (total > 0xffffffffull) throw std::overflow_error("SELL layout exceeds 32-bit offsets");
  }
  S.slice_ptr[S.n_slices] = static_cast<uint32_t>(total);
  S.col.assign(total, -1);
  S.val.assign(total, 0.0);
  for (int t = 0; t < n; ++t) {
    const int r = row_of(t);
    const size_t base = S.slice_ptr[t >> 5] + (t & 31);
    int j = 0;
    for (int p = M.colptr[r]; p < M.colptr[r + 1]; ++p) {
      if (M.val[p] == 0.0) continue;
      S.col[base + 32 * static_cast<size_t>(j)] = M.rowidx[p];
      S.val[base + 32 * static_cast<size_t>(j)] = M.val[p];
      ++j;
    }
    S.nnz += j;
  }
  return S;
}

// ------------------------------------------------------------------ DIA

Dia build_dia(const Csc& M, const std::vector<int>* rows) {
  Dia D;
  const int n = rows ? static_cast<int>(rows->size()) : M.cols;
  auto row_of = [&](int t) { return rows ? (*rows)[t] : t; };
  // distinct offsets col - row over the non-zero entries of the covered rows
  std::vector<int> offs;
  int64_t nnz = 0;
  for (int t = 0; t < n; ++t) {
    const int r = row_of(t);
    for (int p = M.colptr[r]; p < M.colptr[r + 1]; ++p) {
      if (M.val[p] == 0.0) continue;
      ++nnz;
      const int o = M.rowidx[p] - r;
      auto it = std::lower_bound(offs.begin(), offs.end(), o);
      if (it == offs.end() || *it != o) {
        if (static_cast<int>(offs.size()) == kMaxDiag) return D;  // not banded enough
        offs.insert(it, o);
      }
    }
  }
  const int ld = (n + 31) / 32 * 32;
  // refuse when diagonal storage would stream >25% more bytes than SELL (12 B / entry)
  if (8.0 * offs.size() * ld > 1.25 * 12.0 * static_cast<double>(nnz) + 4096.0) return D;
  D.ok = true;
  D.n_rows = n;
  D.n_cols = M.rows;
  D.ld = ld;
  D.n_diag = static_cast<int>(offs.size());
  D.nnz = nnz;
  D.off = offs;
  D.val.assign(static_cast<size_t>(D.n_diag) * ld, 0.0);
  if (rows) D.rows = *rows;
  for (int t = 0; t < n; ++t) {
    const int r = row_of(t);
    for (int p = M.colptr[r]; p < M.colptr[r + 1]; ++p) {
      if (M.val[p] == 0.0) continue;
      const int d = static_cast<int>(std::lower_bound(offs.begin(), offs.end(), M.rowidx[p] - r) - offs.begin());
      D.val[static_cast<size_t>(d) * ld + t] = M.val[p];
    }
  }
  // per-slice occupancy of each diagonal
  const int n_slices = ld / 32;
  std::vector<unsigned short> mask(n_slices, 0);
  int64_t live = 0;
  for (int d = 0; d < D.n_diag; ++d)
    for (int s = 0; s < n_slices; ++s) {
      const double* v = &D.val[static_cast<size_t>(d) * ld + 32 * static_cast<size_t>(s)];
      bool any = false;
      for (int k = 0; k < 32 && !any; ++k) any = (v[k] != 0.0);
      if (any) {
        mask[s] |= static_cast<unsigned short>(1u << d);
        ++live;
      }
    }
  if (live * 10 <= static_cast<int64_t>(D.n_diag) * n_slices * 9) D.mask = std::move(mask);
  return D;
}

Dia build_dia_block(const Csc& M, int row_begin, int n_rows) {
  std::vector<int> rows(n_rows);
  for (int t = 0; t < n_rows; ++t) rows[t] = row_begin + t;
  Dia D = build_dia(M, &rows);
  D.rows.clear();  // local numbering: row t of the block is thread t
  return D;
}

// Rows [row_begin, row_begin + n_rows) of M, local numbering; rows outside [0, M.cols) are empty.
// `offsets` (ascending) fixes the diagonal order, so every rank of a sharded level uses the same
// stencil layout whatever part of the operator its window sees.
Dia build_dia_window(const Csc& M, int row_begin, int n_rows, const std::vector<int>& offsets) {
  Dia D;
  D.ok = true;
  D.n_rows = n_rows;
  D.n_cols = M.rows;
  D.ld = (n_rows + 31) / 32 * 32;
  D.n_diag = static_cast<int>(offsets.size());
  D.off = offsets;
  D.val.assign(static_cast<size_t>(D.n_diag) * D.ld, 0.0);
  for (int t = 0; t < n_rows; ++t) {
    const int r = row_begin + t;
    if (r < 0 || r >= M.cols) continue;
    for (int p = M.colptr[r]; p < M.colptr[r + 1]; ++p) {
      if (M.val[p] == 0.0) continue;
      const int o = M.rowidx[p] - r;
      auto it = std::lower_bound(offsets.begin(), offsets.end(), o);
      if (it == offsets.end() || *it != o) {
        D.ok = false;
        return D;
      }
      D.val[static_cast<size_t>(it - offsets.begin()) * D.ld + t] = M.val[p];
      ++D.nnz;
    }
  }
  return D;
}

// ------------------------------------------------------------------ partition plan

PartitionPlan make_partition_plan(const std::vector<int64_t>& level_sizes,
                                  const std::vector<int>& half_bandwidth, int world,
                                  int64_t min_rows_per_rank, int max_sharded) {
  PartitionPlan P;
  P.world = world;
  P.n_levels = static_cast<int>(level_sizes.size());
  P.n = level_sizes;
  if (world <= 1) return P;
  // deepest prefix of levels that is worth sharding (never the coarsest level)
  int ns = 0;
  while (ns + 1 < P.n_levels && ns < max_sharded && level_sizes[ns] / world >= min_rows_per_rank) ++ns;
  // shrink until every block comfortably contains its halos
  for (; ns > 0; --ns) {
    bool ok = true;
    int ghost = 0;
    for (int l = ns - 1; l >= 0 && ok; --l) {
      ghost = 2 * ghost + 1;
      // the fused legs recompute three chained stencil stages on the ghost rows: 3 (w + 1) + 4
      const int64_t need = std::max<int64_t>(4ll * (half_bandwidth[l] + ghost + 2),
                                             2ll * (3ll * (half_bandwidth[l] + 1) + 4 + ghost)) + (1ll << ns);
      if (level_sizes[l] / world < need) ok = false;
    }
    if (ok) break;
  }
  P.n_sharded = ns;
  if (ns == 0) return P;
  P.start.assign(ns, std::vector<int64_t>(world + 1, 0));
  P.halo_lo.assign(ns, 0);
  P.halo_hi.assign(ns, 0);
  P.ghost.assign(ns, 0);
  const int64_t align = 1ll << ns;
  for (int g = 0; g <= world; ++g) {
    int64_t s0 = (g == world) ? level_sizes[0] : (level_sizes[0] * g / world) / align * align;
    for (int l = 0; l < ns; ++l) {
      P.start[l][g] = (g == world) ? level_sizes[l] : (s0 >> l);
    }
  }
  int ghost = 0;
  for (int l = ns - 1; l >= 0; --l) {
    ghost = 2 * ghost + 1;
    P.ghost[l] = ghost;
    // +2: the fused prolongation sweep evaluates u + P e on the fine halo, which reaches one
    // coarse entry further than the coarse operator's own half-bandwidth
    // 3 (w + 1) + 4 ghost rows on each side let the fused legs (stream_leg.cuh) recompute their
    // three chained stencil stages there; the per-operator kernels need w + 2 (+ ghost above)
    const int fused = 3 * (half_bandwidth[l] + 1) + 4;
    P.halo_lo[l] = std::max(half_bandwidth[l] + 2, fused);
    P.halo_hi[l] = std::max(half_bandwidth[l] + ghost + 2, fused + ghost);
  }
  return P;
}

PartitionPlan make_partition_plan_2d(const std::vector<int64_t>& lines, int world, int64_t min_rows_per_rank) {
  PartitionPlan P;
  P.world = world;
  P.n_levels = static_cast<int>(lines.size());
  for (int64_t m : lines) P.n.push_back(m * m);
  if (world <= 1) return P;
  int ns = 0;
  while (ns + 1 < P.n_levels && P.n[ns] / world >= min_rows_per_rank) ++ns;
  for (; ns > 0; --ns) {
    const int64_t align = 1ll << ns;
    P.start.assign(ns, std::vector<int64_t>(world + 1, 0));
    P.halo_lo.assign(ns, 0);
    P.halo_hi.assign(ns, 0);
    P.ghost.assign(ns, 0);
    bool ok = true;
    int64_t ghost_lines = 0;
    for (int l = ns - 1; l >= 0; --l) {
      ghost_lines = 2 * ghost_lines + 1;
      const int64_t m = lines[l];
      P.ghost[l] = static_cast<int>(ghost_lines * m);
      P.halo_lo[l] = static_cast<int>(m + 2);
      P.halo_hi[l] = static_cast<int>((ghost_lines + 1) * m + 2);
      for (int g = 0; g <= world; ++g) {
        const int64_t y0 = (lines[0] * g / world) / align * align;
        P.start[l][g] = (g == world) ? P.n[l] : (y0 >> l) * m;
      }
      for (int g = 0; g < world; ++g)
        ok = ok && P.start[l][g + 1] - P.start[l][g] >= std::max(P.halo_lo[l], P.halo_hi[l]);
    }
    if (ok) break;
  }
  P.n_sharded = ns;
  if (ns == 0) {
    P.start.clear();
    P.halo_lo.clear();
    P.halo_hi.clear();
    P.ghost.clear();
  }
  return P;
}

// ------------------------------------------------------------------ GS schedule

Schedule gs_schedule(const Csc& M, bool forward) {
  const int n = M.cols;
  std::vector<int> front(n, 0);
  int n_fronts = 0;
  auto visit = [&](int k) {
    int f = 0;
    for (int p = M.colptr[k]; p < M.colptr[k + 1]; ++p) {
      const int j = M.rowidx[p];
      if (M.val[p] == 0.0) continue;
      if (forward ? (j < k) : (j > k)) f = std::max(f, front[j] + 1);
    }
    front[k] = f;
    n_fronts = std::max(n_fronts, f + 1);
  };
  if (forward)
    for (int k = 0; k < n; ++k) visit(k);
  else
    for (int k = n - 1; k >= 0; --k) visit(k);
  Schedule S;
  S.front_ptr.assign((size_t)n_fronts + 1, 0);
  for (int k = 0; k < n; ++k) S.front_ptr[front[k] + 1]++;
  for (int f = 0; f < n_fronts; ++f) {
    S.max_width = std::max(S.max_width, S.front_ptr[f + 1]);
    S.front_ptr[f + 1] += S.front_ptr[f];
  }
  S.order.resize(n);
  std::vector<int> cursor(S.front_ptr.begin(), S.front_ptr.end() - 1);
  if (forward)
    for (int k = 0; k < n; ++k) S.order[cursor[front[k]]++] = k;
  else
    for (int k = n - 1; k >= 0; --k) S.order[cursor[front[k]]++] = k;
  return S;
}

}  // namespace amgb
