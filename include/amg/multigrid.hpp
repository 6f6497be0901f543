// Mirror of include/amg/multigrid.hpp: AMG::Multigrid (:22-365) with the reference's
// constructor signature, vcycle(), solve(), getters and display flag; the hierarchy lives
// on the GPU (amgb_hierarchy) and one vcycle() is one CUDA-graph replay.  Beyond the
// reference, the iteration count and the error history are available programmatically
// (the reference only prints them).
#pragma once
#include <iostream>
#include <vector>

#include "common.hpp"
#include "grid.hpp"
#include "interpolator.hpp"
#include "smoother.hpp"

namespace AMG {

template <class EleType>
class Multigrid {
 private:
  InterpolatorBase<EleType>* interpolator;  // non-owning, like the reference (:29-31)
  SmootherBase<EleType>* smoother;
  amgb_hierarchy* h{nullptr};
  size_t n_levels;
  EleType tolerance;
  size_t compute_error_every_n_iters;
  size_t n_iters;
  bool display_error{false};
  // host copies handed out by reference from the getters
  mutable std::vector<SparseMatrixT<EleType>> level_to_coefficient_matrix;
  mutable std::vector<VectorT<EleType>> level_to_soln;
  mutable std::vector<VectorT<EleType>> level_to_rhs;
  size_t iters_done_{0};
  EleType last_error_{100};

 public:
  ~Multigrid() {
    if (h) amgb_hierarchy_destroy(h);
  }
  Multigrid() = delete;
  Multigrid(const Multigrid&) = delete;
  Multigrid& operator=(const Multigrid&) = delete;

  Multigrid(InterpolatorBase<EleType>* interpolator_, SmootherBase<EleType>* smoother_,
            const SparseMatrixT<EleType>& A, const VectorT<EleType>& b, size_t n_levels_,
            EleType tolerance_ = 1e-9, size_t compute_error_every_n_iters_ = 10, size_t n_iters_ = 100)
      : interpolator(interpolator_),
        smoother(smoother_),
        n_levels(n_levels_),
        tolerance(tolerance_),
        compute_error_every_n_iters(compute_error_every_n_iters_),
        n_iters(n_iters_) {
    static_assert(sizeof(EleType) == sizeof(double), "the device path is fp64 only");
    amgb_options opt;
    amgb_options_default(&opt);
    opt.n_levels = (int)n_levels;
    opt.tolerance = tolerance;
    opt.compute_error_every_n_iters = (int64_t)compute_error_every_n_iters;
    opt.n_iters = (int64_t)n_iters;
    // the two reference checks (multigrid.hpp:165-178) come first, inside the C ABI
    if (compute_error_every_n_iters <= n_iters && (size_t)A.rows() == (size_t)b.rows()) {
      if (!smoother || smoother->device_kind() < 0)
        throw std::invalid_argument("the GPU driver needs a SparseGaussSeidel, DampedJacobi, LineGaussSeidel or "
                                    "MulticolorGaussSeidel smoother");
      if (!interpolator || interpolator->device_transfer() < 0)
        throw std::invalid_argument("the GPU driver applies the operators of LinearInterpolator, "
                                    "BilinearInterpolator2D or SmoothedAggregationInterpolator");
    }
    if (interpolator && interpolator->device_transfer() >= 0) opt.transfer = interpolator->device_transfer();
    const bool sa = opt.transfer == AMGB_TRANSFER_SMOOTHED_AGGREGATION;
    if (sa) opt.strength = interpolator->device_strength();
    if (smoother && smoother->device_kind() >= 0) {
      opt.smoother = smoother->device_kind();
      opt.smoother_iters = (int64_t)smoother->n_iters;
      opt.omega = smoother->device_omega();
      opt.lines = smoother->device_lines();
    }
    if (!A.isCompressed()) throw std::invalid_argument("A must be compressed (makeCompressed())");
    detail::check(amgb_hierarchy_create((int)A.rows(), (int)A.cols(), A.outerIndexPtr(), A.innerIndexPtr(),
                                        A.valuePtr(), b.data(), (int64_t)b.rows(), &opt, &h));
    n_levels = (size_t)amgb_hierarchy_n_levels(h);  // smoothed aggregation: n_levels_ is a cap
    level_to_coefficient_matrix.resize(n_levels);
    level_to_soln.resize(n_levels);
    level_to_rhs.resize(n_levels);
    // fill the interpolator's slots 0..L-2 like the reference's constructor does (:211-218)
    for (size_t level = 1; level < n_levels; ++level) {
      if (sa) fill_transfer(level - 1);
      else interpolator->make_operators(get_n_dofs(level - 1), get_n_dofs(level), level - 1);
    }
  }

  void vcycle() { detail::check(amgb_vcycle(h)); }  // multigrid.hpp:263-305

  const VectorT<EleType>& solve() {  // multigrid.hpp:311-337
    int64_t it = 0;
    double err = 100;
    detail::check(amgb_solve(h, &it, &err));
    iters_done_ = (size_t)it;
    last_error_ = err;
    if (display_error) {
      const std::vector<EleType> hist = error_history();
      for (size_t k = 0; k < hist.size(); ++k)
        std::cout << "Iter: " << (k + 1) * compute_error_every_n_iters << " | Error: " << hist[k] << std::endl;
    }
    if (err <= tolerance)
      std::cout << "AMG converged after " << it << " iterations." << std::endl;
    else
      std::cout << "AMG did not converge after " << it << " iterations." << std::endl;
    return get_soln(0);
  }

  const SparseMatrixT<EleType>& get_coefficient_matrix(size_t level) const {
    auto& M = level_to_coefficient_matrix[level];
    if (M.rows() == 0) {
      const int64_t n = amgb_hierarchy_n_dofs(h, (int)level), nnz = amgb_hierarchy_nnz(h, (int)level);
      std::vector<int> outer(n + 1), inner(nnz);
      std::vector<double> val(nnz);
      detail::check(amgb_hierarchy_get_matrix(h, (int)level, outer.data(), inner.data(), val.data()));
#if AMGB_HAVE_EIGEN
      M = Eigen::Map<const Eigen::SparseMatrix<double>>((int)n, (int)n, nnz, outer.data(), inner.data(),
                                                        val.data());
#else
      M = SparseMatrixT<EleType>((int)n, (int)n, std::move(outer), std::move(inner), std::move(val));
#endif
    }
    return M;
  }
  const VectorT<EleType>& get_soln(size_t level) const {
    auto& u = level_to_soln[level];
    u.resize((size_t)amgb_hierarchy_n_dofs(h, (int)level));
    detail::check(amgb_hierarchy_get_soln(h, (int)level, u.data()));
    return u;
  }
  const VectorT<EleType>& get_rhs(size_t level) const {
    auto& f = level_to_rhs[level];
    f.resize((size_t)amgb_hierarchy_n_dofs(h, (int)level));
    detail::check(amgb_hierarchy_get_rhs(h, (int)level, f.data()));
    return f;
  }
  const size_t get_n_dofs(size_t level) const { return (size_t)amgb_hierarchy_n_dofs(h, (int)level); }
  const EleType get_tolerance() const { return tolerance; }

  void display_error_on() { display_error = true; }
  // the reference sets the flag to true here as well (multigrid.hpp:361-364); this mirror
  // does what the name says
  void display_error_off() { display_error = false; }

  // ---- beyond the reference ----
  size_t iterations_done() const { return iters_done_; }
  EleType last_error() const { return last_error_; }
  std::vector<EleType> error_history() const {
    const int64_t n = amgb_hierarchy_error_history(h, nullptr, 0);
    std::vector<EleType> out((size_t)n);
    if (n) amgb_hierarchy_error_history(h, out.data(), n);
    return out;
  }
  // Conjugate gradients preconditioned by one V-cycle (the use the reference's README names,
  // README.md:127); stops at ||r||_2 / ||b||_2 <= rel_tol or after max_iters iterations.
  const VectorT<EleType>& solve_pcg(EleType rel_tol, size_t max_iters = 1000) {
    int64_t it = 0;
    double rel = 0;
    detail::check(amgb_solve_pcg(h, rel_tol, (int64_t)max_iters, &it, &rel));
    iters_done_ = (size_t)it;
    last_error_ = rel;
    return get_soln(0);
  }
  // Restarted GMRES(restart) right-preconditioned by one V-cycle, for unsymmetric A as well (amgb.h,
  // amgb_solve_gmres); iterations_done() counts Arnoldi steps, last_error() is the true relative residual.
  const VectorT<EleType>& solve_gmres(EleType rel_tol, int restart = 30, size_t max_iters = 1000) {
    int64_t it = 0;
    double rel = 0;
    detail::check(amgb_solve_gmres(h, rel_tol, restart, (int64_t)max_iters, &it, &rel));
    iters_done_ = (size_t)it;
    last_error_ = rel;
    return get_soln(0);
  }
  amgb_hierarchy* handle() { return h; }
  size_t get_n_levels() const { return n_levels; }

 private:
  // P of `level` as the hierarchy built it, and R = P^T (an index permutation), into the interpolator
  void fill_transfer(size_t level) {
    const int nf = (int)get_n_dofs(level), nc = (int)get_n_dofs(level + 1);
    int64_t nnz = 0;
    detail::check(amgb_hierarchy_get_transfer(h, (int)level, &nnz, nullptr, nullptr, nullptr));
    std::vector<int> Pc(nc + 1), Pr(nnz), Rc(nf + 1, 0), Rr(nnz);
    std::vector<double> Pv(nnz), Rv(nnz);
    detail::check(amgb_hierarchy_get_transfer(h, (int)level, &nnz, Pc.data(), Pr.data(), Pv.data()));
    for (int64_t p = 0; p < nnz; ++p) Rc[Pr[p] + 1]++;
    for (int i = 0; i < nf; ++i) Rc[i + 1] += Rc[i];
    std::vector<int> cursor(Rc.begin(), Rc.end() - 1);
    for (int J = 0; J < nc; ++J)
      for (int p = Pc[J]; p < Pc[J + 1]; ++p) {
        const int q = cursor[Pr[p]]++;
        Rr[q] = J;
        Rv[q] = Pv[p];
      }
#if AMGB_HAVE_EIGEN
    SparseMatrixT<EleType> P = Eigen::Map<const Eigen::SparseMatrix<double>>(nf, nc, nnz, Pc.data(), Pr.data(),
                                                                             Pv.data());
    SparseMatrixT<EleType> R = Eigen::Map<const Eigen::SparseMatrix<double>>(nc, nf, nnz, Rc.data(), Rr.data(),
                                                                             Rv.data());
#else
    SparseMatrixT<EleType> P(nf, nc, std::move(Pc), std::move(Pr), std::move(Pv));
    SparseMatrixT<EleType> R(nc, nf, std::move(Rc), std::move(Rr), std::move(Rv));
#endif
    interpolator->set_level_to_P(level, P);
    interpolator->set_level_to_R(level, R);
  }
};

}  // namespace AMG
