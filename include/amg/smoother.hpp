// Mirror of include/amg/smoother.hpp: SmootherBase (:18-66) and SparseGaussSeidel
// (:86-216) with the same public fields, constructors and smooth() signature; smooth()
// forwards the CSC arrays and the vectors to the GPU through the C ABI (amgb.h).
// DampedJacobi and MulticolorGaussSeidel are the partitionable smoothers the B200 build
// adds.  The reference's Jacobi / SuccessiveOverRelaxation test smoothers (:223-373) are not
// on the V-cycle path (dense O(N^2) loops, unusable beyond toy sizes); they are provided as
// HOST-ONLY classes with the reference's names, constructors, validation and update formulas
// so that code written against the reference (test/testlib.cpp:65-107) compiles unchanged
// against this include directory.  The GPU Multigrid driver refuses them (device_kind() < 0).
#pragma once
#include <iostream>
#include <string>
#include <vector>

#include "common.hpp"

namespace AMG {

template <class EleType>
class SmootherBase {
 public:
  EleType tolerance{1e-9};
  size_t compute_error_every_n_iters{100};
  size_t n_iters{1};

  SmootherBase() {}
  SmootherBase(size_t n_iters_) : n_iters(n_iters_) {}
  SmootherBase(double tolerance_, size_t compute_error_every_n_iters_, size_t n_iters_)
      : tolerance(tolerance_), compute_error_every_n_iters(compute_error_every_n_iters_), n_iters(n_iters_) {}
  virtual ~SmootherBase() {}

  virtual void smooth(const SparseMatrixT<EleType>& A, VectorT<EleType>& u, const VectorT<EleType>& b) = 0;

  // Which device smoother the GPU Multigrid driver runs for this object
  // (AMGB_SMOOTHER_*), or -1 for a host-only user smoother the driver cannot use.
  virtual int device_kind() const { return -1; }
  virtual double device_omega() const { return 2.0 / 3.0; }
  // AMGB_LINES_* of a line smoother (AMGB_SMOOTHER_LINE_GS)
  virtual int device_lines() const { return AMGB_LINES_X; }
};

template <class EleType>
class SparseGaussSeidel : public SmootherBase<EleType> {
 public:
  using SmootherBase<EleType>::SmootherBase;
  size_t iters_done{0};     // beyond the reference, which only prints these
  EleType last_error{100};
  int mode{AMGB_GS_AUTO};

  SparseGaussSeidel() {  // smoother.hpp:183-187
    this->tolerance = 1e-9;
    this->compute_error_every_n_iters = 0;
    this->n_iters = 1;
  }
  void smooth(const SparseMatrixT<EleType>& A, VectorT<EleType>& u, const VectorT<EleType>& b) override {
    int64_t it = 0;
    double err = 100;
    detail::check(amgb_smooth_gs(detail::MirrorCache::instance().get(A), u.data(), b.data(), this->tolerance,
                                 (int64_t)this->compute_error_every_n_iters, (int64_t)this->n_iters, mode, &it,
                                 &err));
    iters_done = (size_t)it;
    last_error = err;
    if (this->compute_error_every_n_iters != 0) {  // smoother.hpp:205-212
      if (err <= this->tolerance)
        std::cout << "SPGS converged after " << it << " iterations." << std::endl;
      else
        std::cout << "SPGS did not converge after " << it << " iterations." << std::endl;
    }
  }
  int device_kind() const override { return AMGB_SMOOTHER_GS; }
};

// u <- u + omega D^-1 (f - A u); n_iters sweeps per smooth() call.
template <class EleType>
class DampedJacobi : public SmootherBase<EleType> {
  double omega_{2.0 / 3.0};

 public:
  DampedJacobi(double omega = 2.0 / 3.0, size_t n_sweeps = 2) : SmootherBase<EleType>(n_sweeps), omega_(omega) {
    if (omega <= 0 || omega > 2)
      throw std::invalid_argument("`omega` must be in (0, 2] but got omega=" + std::to_string(omega));
  }
  void smooth(const SparseMatrixT<EleType>& A, VectorT<EleType>& u, const VectorT<EleType>& b) override {
    detail::check(amgb_smooth_jacobi(detail::MirrorCache::instance().get(A), u.data(), b.data(), omega_,
                                     (int64_t)this->n_iters));
  }
  int device_kind() const override { return AMGB_SMOOTHER_JACOBI; }
  double device_omega() const override { return omega_; }
};

// greedy multicolour symmetric Gauss-Seidel (red-black on the five-point level)
template <class EleType>
class MulticolorGaussSeidel : public SmootherBase<EleType> {
 public:
  MulticolorGaussSeidel(size_t n_iters_ = 1) : SmootherBase<EleType>(n_iters_) {}
  void smooth(const SparseMatrixT<EleType>& A, VectorT<EleType>& u, const VectorT<EleType>& b) override {
    detail::check(amgb_smooth_color_gs(detail::MirrorCache::instance().get(A), u.data(), b.data(),
                                       (int64_t)this->n_iters));
  }
  int device_kind() const override { return AMGB_SMOOTHER_COLOR_GS; }
};

// zebra line Gauss-Seidel on an m x m grid operator (amgb.h, AMGB_SMOOTHER_LINE_GS): n_iters x (forward
// half then backward half) per smooth() call; the GPU Multigrid driver needs BilinearInterpolator2D
template <class EleType>
class LineGaussSeidel : public SmootherBase<EleType> {
  int lines_{AMGB_LINES_X};

 public:
  LineGaussSeidel(size_t n_iters_ = 1, int lines = AMGB_LINES_X) : SmootherBase<EleType>(n_iters_), lines_(lines) {
    if (lines != AMGB_LINES_X && lines != AMGB_LINES_Y && lines != AMGB_LINES_ALTERNATING)
      throw std::invalid_argument("`lines` must be AMGB_LINES_X, AMGB_LINES_Y or AMGB_LINES_ALTERNATING but got " +
                                  std::to_string(lines));
  }
  void smooth(const SparseMatrixT<EleType>& A, VectorT<EleType>& u, const VectorT<EleType>& b) override {
    detail::check(amgb_smooth_line_gs(detail::MirrorCache::instance().get(A), u.data(), b.data(),
                                      (int64_t)this->n_iters, lines_));
  }
  int device_kind() const override { return AMGB_SMOOTHER_LINE_GS; }
  int device_lines() const override { return lines_; }
};

namespace detail {
// Rows of a compressed ColMajor matrix (host): row i = the entries A(i, j) in ascending j.
// The reference walks A.coeff(i, j) over ALL j (smoother.hpp:247-253, :347-357); the absent
// entries add exact zeros, so walking the stored ones in the same order gives the same sums.
template <class Mat, class T>
struct HostRows {
  std::vector<long> ptr;
  std::vector<int> col;
  std::vector<T> val;
  explicit HostRows(const Mat& A) {
    const long n = (long)A.rows(), m = (long)A.cols();
    const int* cp = A.outerIndexPtr();
    const int* ri = A.innerIndexPtr();
    const auto* v = A.valuePtr();
    ptr.assign((size_t)n + 1, 0);
    for (long p = 0; p < cp[m]; ++p) ++ptr[(size_t)ri[p] + 1];
    for (long i = 0; i < n; ++i) ptr[(size_t)i + 1] += ptr[(size_t)i];
    col.resize((size_t)cp[m]);
    val.resize((size_t)cp[m]);
    std::vector<long> fill(ptr.begin(), ptr.end() - 1);
    for (long j = 0; j < m; ++j)
      for (long p = cp[j]; p < cp[j + 1]; ++p) {
        const long q = fill[(size_t)ri[p]]++;
        col[(size_t)q] = (int)j;
        val[(size_t)q] = (T)v[p];
      }
  }
};
}  // namespace detail

// Host-only counterpart of the reference's `Jacobi` (smoother.hpp:223-263).  As in the
// reference, u[i] is overwritten inside the row loop, i.e. the method is a forward
// Gauss-Seidel sweep; the error is the device rss every compute_error_every_n_iters sweeps.
template <class EleType>
class Jacobi : public SmootherBase<EleType> {
 public:
  using SmootherBase<EleType>::SmootherBase;
  Jacobi() {}
  void smooth(const SparseMatrixT<EleType>& A, VectorT<EleType>& u, const VectorT<EleType>& b) override {
    const detail::HostRows<SparseMatrixT<EleType>, EleType> R(A);
    const size_t ndofs = (size_t)b.size();
    size_t iter = 0;
    EleType error = 100;
    while (iter < this->n_iters && error > this->tolerance) {
      for (size_t i = 0; i < ndofs; ++i) {
        EleType sigma = 0, aii = 0;
        for (long p = R.ptr[i]; p < R.ptr[i + 1]; ++p) {
          if ((size_t)R.col[(size_t)p] == i) aii = R.val[(size_t)p];
          else sigma += R.val[(size_t)p] * u[(size_t)R.col[(size_t)p]];
        }
        u[i] = (b[i] - sigma) / aii;
      }
      iter += 1;
      if (this->compute_error_every_n_iters != 0 && iter % this->compute_error_every_n_iters == 0)
        error = rss(A, u, b);
    }
  }
};

// Host-only counterpart of the reference's `SuccessiveOverRelaxation` (smoother.hpp:265-373):
// omega in [0, 2] validated by the constructors that take it (std::invalid_argument, :286-293),
// u_i <- u_i + omega (u_i^GS - u_i).
template <class EleType>
class SuccessiveOverRelaxation : public SmootherBase<EleType> {
  double omega{1.0};
  void validate_omega() {
    if (omega > 2 || omega < 0)
      throw std::invalid_argument("`omega` must be in [0, 2] but got omega=" + std::to_string(omega) + "\n");
  }

 public:
  using SmootherBase<EleType>::SmootherBase;
  SuccessiveOverRelaxation() {}
  SuccessiveOverRelaxation(double omega_) : omega(omega_) { validate_omega(); }
  SuccessiveOverRelaxation(double omega_, double tolerance_, size_t compute_error_every_n_iters_, size_t n_iters_)
      : SmootherBase<EleType>(tolerance_, compute_error_every_n_iters_, n_iters_), omega(omega_) {
    validate_omega();
  }
  void smooth(const SparseMatrixT<EleType>& A, VectorT<EleType>& u, const VectorT<EleType>& b) override {
    const detail::HostRows<SparseMatrixT<EleType>, EleType> R(A);
    const size_t ndofs = (size_t)b.size();
    size_t iter = 0;
    EleType error = 100;
    while (iter < this->n_iters && error > this->tolerance) {
      for (size_t i = 0; i < ndofs; ++i) {
        EleType below = 0, above = 0, aii = 0;
        for (long p = R.ptr[i]; p < R.ptr[i + 1]; ++p) {
          const size_t j = (size_t)R.col[(size_t)p];
          if (j < i) below += R.val[(size_t)p] * u[j];
          else if (j > i) above += R.val[(size_t)p] * u[j];
          else aii = R.val[(size_t)p];
        }
        const EleType gs = (b[i] - below - above) / aii;
        const EleType uk = u[i];
        u[i] = uk + omega * (gs - uk);
      }
      iter += 1;
      if (this->compute_error_every_n_iters != 0 && iter % this->compute_error_every_n_iters == 0)
        error = rss(A, u, b);
    }
  }
};

}  // namespace AMG
