// Mirror of include/amg/interpolator.hpp: InterpolatorBase (:15-87) keeps per-level P / R
// with the same getters / setters and a virtual make_operators; LinearInterpolator
// (:98-141) builds the reference's operators (bit-exact integer maps) through the C ABI.
// restriction() / prolongation() stay non-virtual members returning a new vector, as in the
// reference (:52-68), and apply the STORED operators: matrix-free on the GPU when those are the
// linear-interpolation operators, through the generic device SpMV otherwise.
#pragma once
#include <stdexcept>
#include <vector>

#include "compat.hpp"

namespace AMG {
namespace detail {
// P (n_h x n_H, compressed CSC) is exactly LinearInterpolator's operator: column j holds rows
// 2j, 2j+1, 2j+2 (those below n_h) with values .5, 1, .5 (interpolator.hpp:106-141)
template <class Mat>
inline bool is_linear_prolongation(const Mat& P) {
  if (!P.isCompressed()) return false;
  const long n_h = (long)P.rows(), n_H = (long)P.cols();
  const int* cp = P.outerIndexPtr();
  const int* ri = P.innerIndexPtr();
  const auto* v = P.valuePtr();
  static const double w[3] = {0.5, 1.0, 0.5};
  long p = 0;
  for (long j = 0; j < n_H; ++j) {
    if (cp[j] != p) return false;
    for (int k = 0; k < 3; ++k) {
      if (2 * j + k >= n_h) continue;
      if (p >= (long)P.nonZeros() || ri[p] != 2 * j + k || v[p] != w[k]) return false;
      ++p;
    }
  }
  return cp[n_H] == p && p == (long)P.nonZeros();
}
// R (n_H x n_h) is its transpose: column k holds row (k-1)/2 with 1 for odd k, rows k/2-1 and
// k/2 (those inside [0, n_H)) with .5 for even k
template <class Mat>
inline bool is_linear_restriction(const Mat& R) {
  if (!R.isCompressed()) return false;
  const long n_H = (long)R.rows(), n_h = (long)R.cols();
  const int* cp = R.outerIndexPtr();
  const int* ri = R.innerIndexPtr();
  const auto* v = R.valuePtr();
  long p = 0;
  for (long k = 0; k < n_h; ++k) {
    if (cp[k] != p) return false;
    if (k & 1) {
      const long J = (k - 1) / 2;
      if (J < n_H) {
        if (p >= (long)R.nonZeros() || ri[p] != J || v[p] != 1.0) return false;
        ++p;
      }
    } else {
      for (long J = k / 2 - 1; J <= k / 2; ++J) {
        if (J < 0 || J >= n_H) continue;
        if (p >= (long)R.nonZeros() || ri[p] != J || v[p] != 0.5) return false;
        ++p;
      }
    }
  }
  return cp[n_h] == p && p == (long)R.nonZeros();
}
}  // namespace detail

template <class EleType>
class InterpolatorBase {
 private:
  std::vector<SparseMatrixT<EleType>> level_to_P;
  std::vector<SparseMatrixT<EleType>> level_to_R;

 public:
  InterpolatorBase(size_t n_levels) {  // interpolator.hpp:22-26
    level_to_P.resize(n_levels - 1);
    level_to_R.resize(n_levels - 1);
  }
  InterpolatorBase() {}
  virtual ~InterpolatorBase() {}

  virtual void make_operators(size_t n_h_dofs, size_t n_H_dofs, size_t level) = 0;
  // AMGB_TRANSFER_* of the device kernels that apply this interpolator's operators matrix-free
  // (-1: none, the GPU driver cannot run it)
  virtual int device_transfer() const { return -1; }
  // strength threshold theta of AMGB_TRANSFER_SMOOTHED_AGGREGATION (the library default for the others)
  virtual double device_strength() const { return 0.08; }
  // true when P is the reference's linear interpolation
  bool is_linear_interpolation() const { return device_transfer() == AMGB_TRANSFER_LINEAR; }

  // :52-56 and :64-68 -- get_P(level) * v and get_R(level) * v with the operators that are
  // STORED, whoever put them there (make_operators of any subclass, set_level_to_P/R).  When the
  // stored operator is the reference's linear interpolation (checked entry by entry on the
  // host, O(nnz)) the matrix-free device kernel runs; any other operator goes through the
  // generic device SpMV, in Eigen's summation order.
  VectorT<EleType> prolongation(const VectorT<EleType>& v, size_t level) {
    const auto& P = get_P(level);
    VectorT<EleType> result((size_t)P.rows());
    if (detail::is_linear_prolongation(P))
      detail::check(amgb_linear_prolong((int64_t)P.rows(), (int64_t)P.cols(), v.data(), result.data()));
    else
      detail::check(amgb_csc_spmv((int)P.rows(), (int)P.cols(), P.outerIndexPtr(), P.innerIndexPtr(),
                                  P.valuePtr(), v.data(), result.data()));
    return result;
  }
  VectorT<EleType> restriction(const VectorT<EleType>& v, size_t level) {
    const auto& R = get_R(level);
    VectorT<EleType> result((size_t)R.rows());
    if (detail::is_linear_restriction(R))
      detail::check(amgb_linear_restrict((int64_t)R.cols(), (int64_t)R.rows(), v.data(), result.data()));
    else
      detail::check(amgb_csc_spmv((int)R.rows(), (int)R.cols(), R.outerIndexPtr(), R.innerIndexPtr(),
                                  R.valuePtr(), v.data(), result.data()));
    return result;
  }
  const SparseMatrixT<EleType>& get_P(size_t level) const { return level_to_P[level]; }
  const SparseMatrixT<EleType>& get_R(size_t level) const { return level_to_R[level]; }
  void set_level_to_P(size_t level, SparseMatrixT<EleType>& P) { level_to_P[level] = P; }
  void set_level_to_R(size_t level, SparseMatrixT<EleType>& R) { level_to_R[level] = R; }
};

template <class EleType>
class LinearInterpolator : public InterpolatorBase<EleType> {
 public:
  using InterpolatorBase<EleType>::InterpolatorBase;

  void make_operators(size_t n_h_dofs, size_t n_H_dofs, size_t level) override {  // :106-141
    const int64_t nnz = amgb_interp_nnz((int64_t)n_h_dofs, (int64_t)n_H_dofs);
    std::vector<int> Pc(n_H_dofs + 1), Pr(nnz), Rc(n_h_dofs + 1), Rr(nnz);
    std::vector<double> Pv(nnz), Rv(nnz);
    detail::check(amgb_interp_make_operators((int64_t)n_h_dofs, (int64_t)n_H_dofs, Pc.data(), Pr.data(),
                                             Pv.data(), Rc.data(), Rr.data(), Rv.data()));
#if AMGB_HAVE_EIGEN
    SparseMatrixT<EleType> P = Eigen::Map<const Eigen::SparseMatrix<double>>(
        (int)n_h_dofs, (int)n_H_dofs, nnz, Pc.data(), Pr.data(), Pv.data());
    SparseMatrixT<EleType> R = Eigen::Map<const Eigen::SparseMatrix<double>>(
        (int)n_H_dofs, (int)n_h_dofs, nnz, Rc.data(), Rr.data(), Rv.data());
#else
    SparseMatrixT<EleType> P((int)n_h_dofs, (int)n_H_dofs, std::move(Pc), std::move(Pr), std::move(Pv));
    SparseMatrixT<EleType> R((int)n_H_dofs, (int)n_h_dofs, std::move(Rc), std::move(Rr), std::move(Rv));
#endif
    this->set_level_to_P(level, P);
    this->set_level_to_R(level, R);
  }
  int device_transfer() const override { return AMGB_TRANSFER_LINEAR; }
};

// Bilinear interpolation on an m x m grid of DOFs numbered k = y*m + x (no reference counterpart):
// P = P1 (x) P1 with LinearInterpolator's 1-D pattern P1, m_H = m_h / 2, R = P^T.  The 2-D
// coarsening under which the V-cycle converges independently of the grid size on 2-D problems.
template <class EleType>
class BilinearInterpolator2D : public InterpolatorBase<EleType> {
 public:
  using InterpolatorBase<EleType>::InterpolatorBase;

  void make_operators(size_t n_h_dofs, size_t n_H_dofs, size_t level) override {
    const int64_t m_h = lines(n_h_dofs), m_H = lines(n_H_dofs);
    if (m_h < 0 || m_H < 0 || m_H != amgb_bilinear_coarse_lines(m_h))
      throw std::invalid_argument("BilinearInterpolator2D: " + std::to_string(n_h_dofs) + " -> " +
                                  std::to_string(n_H_dofs) + " DOFs are not m^2 -> (m / 2)^2");
    const int64_t nnz = amgb_bilinear_nnz(m_h, m_H);
    std::vector<int> Pc(n_H_dofs + 1), Pr(nnz), Rc(n_h_dofs + 1), Rr(nnz);
    std::vector<double> Pv(nnz), Rv(nnz);
    detail::check(amgb_bilinear_make_operators(m_h, m_H, Pc.data(), Pr.data(), Pv.data(), Rc.data(), Rr.data(),
                                               Rv.data()));
#if AMGB_HAVE_EIGEN
    SparseMatrixT<EleType> P = Eigen::Map<const Eigen::SparseMatrix<double>>(
        (int)n_h_dofs, (int)n_H_dofs, nnz, Pc.data(), Pr.data(), Pv.data());
    SparseMatrixT<EleType> R = Eigen::Map<const Eigen::SparseMatrix<double>>(
        (int)n_H_dofs, (int)n_h_dofs, nnz, Rc.data(), Rr.data(), Rv.data());
#else
    SparseMatrixT<EleType> P((int)n_h_dofs, (int)n_H_dofs, std::move(Pc), std::move(Pr), std::move(Pv));
    SparseMatrixT<EleType> R((int)n_H_dofs, (int)n_h_dofs, std::move(Rc), std::move(Rr), std::move(Rv));
#endif
    this->set_level_to_P(level, P);
    this->set_level_to_R(level, R);
  }
  int device_transfer() const override { return AMGB_TRANSFER_BILINEAR_2D; }

 private:
  static int64_t lines(size_t n) {  // m with m * m == n, else -1
    int64_t m = 0;
    while ((m + 1) * (m + 1) <= (int64_t)n) ++m;
    return m * m == (int64_t)n ? m : -1;
  }
};

// Smoothed-aggregation coarsening (no reference counterpart; include/amgb.h,
// AMGB_TRANSFER_SMOOTHED_AGGREGATION): aggregates of strongly coupled rows (threshold theta), P smoothed by
// one damped-Jacobi step.  It needs no grid.  n_levels is a cap: the hierarchy coarsens while a level has
// more than 200 rows, and stops at a coarse level whose aggregation does not reduce it.  The aggregation depends on A, so Multigrid builds the operators and fills the P and
// R slots; make_operators, which only knows the sizes, throws std::logic_error.
template <class EleType>
class SmoothedAggregationInterpolator : public InterpolatorBase<EleType> {
 public:
  explicit SmoothedAggregationInterpolator(size_t n_levels, double theta = 0.08)
      : InterpolatorBase<EleType>(n_levels), theta_(theta) {}

  void make_operators(size_t, size_t, size_t) override {
    throw std::logic_error("SmoothedAggregationInterpolator: the aggregation depends on A, so Multigrid builds "
                           "the operators (make_operators cannot build them from the level sizes)");
  }
  int device_transfer() const override { return AMGB_TRANSFER_SMOOTHED_AGGREGATION; }
  double strength() const { return theta_; }
  double device_strength() const override { return theta_; }

 private:
  double theta_;
};

}  // namespace AMG
