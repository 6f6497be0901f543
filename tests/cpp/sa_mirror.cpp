// C++ check of SmoothedAggregationInterpolator in the include/amg mirror headers: make_operators
// refuses to build operators from sizes alone, and (on the GPU) a Multigrid that builds the
// smoothed-aggregation hierarchy of a rectangular grid operator, fills the interpolator's P and R
// slots from it and converges.
#include <cmath>
#include <cstdio>
#include <stdexcept>
#include <string>
#include <vector>

#include <amg/common.hpp>
#include <amg/grid.hpp>
#include <amg/interpolator.hpp>
#include <amg/multigrid.hpp>
#include <amg/smoother.hpp>

using Mat = AMG::SparseMatrixT<double>;
using Vec = AMG::VectorT<double>;

static int g_failed = 0;
#define CHECK(cond)                                                     \
  do {                                                                  \
    if (!(cond)) {                                                      \
      std::printf("CHECK FAILED %s:%d: %s\n", __FILE__, __LINE__, #cond); \
      ++g_failed;                                                       \
    }                                                                   \
  } while (0)

// 5-point Poisson on an nx x ny grid (x fastest), compressed CSC
static Mat rectangular_poisson(int nx, int ny) {
  const int n = nx * ny;
  std::vector<int> outer(n + 1, 0), inner;
  std::vector<double> val;
  for (int k = 0; k < n; ++k) {
    const int x = k % nx, y = k / nx;
    auto put = [&](int r, double v) {
      inner.push_back(r);
      val.push_back(v);
    };
    if (y > 0) put(k - nx, 1.0);
    if (x > 0) put(k - 1, 1.0);
    put(k, -4.0);
    if (x + 1 < nx) put(k + 1, 1.0);
    if (y + 1 < ny) put(k + nx, 1.0);
    outer[k + 1] = (int)inner.size();
  }
#if AMGB_HAVE_EIGEN
  return Eigen::Map<const Eigen::SparseMatrix<double>>(n, n, (int)inner.size(), outer.data(), inner.data(), val.data());
#else
  return Mat(n, n, std::move(outer), std::move(inner), std::move(val));
#endif
}

int main(int argc, char** argv) {
  AMG::SmoothedAggregationInterpolator<double> sa(4, 0.1);
  CHECK(sa.device_transfer() == AMGB_TRANSFER_SMOOTHED_AGGREGATION);
  CHECK(sa.strength() == 0.1);
  bool threw = false;
  try {
    sa.make_operators(100, 25, 0);
  } catch (const std::logic_error&) {
    threw = true;
  }
  CHECK(threw);
  if (argc > 1 && std::string(argv[1]) == "gpu") {
    const int nx = 150, ny = 60;
    Mat A = rectangular_poisson(nx, ny);
    Vec b(nx * ny);
    for (int i = 0; i < nx * ny; ++i) b[i] = std::sin(0.01 * i);
    AMG::SmoothedAggregationInterpolator<double> interp(20);
    AMG::DampedJacobi<double> jac(2.0 / 3.0, 2);
    AMG::Multigrid<double> mg(&interp, &jac, A, b, 20, 1e-9, 1, 100);
    const size_t L = mg.get_n_levels();
    CHECK(L >= 3 && L < 20);
    CHECK(amgb_hierarchy_n_levels(mg.handle()) == (int)L);
    CHECK(mg.get_n_dofs(L - 1) <= 200 && mg.get_n_dofs(L - 2) > 200);
    for (size_t l = 0; l + 1 < L; ++l) {
      CHECK((size_t)interp.get_P(l).rows() == mg.get_n_dofs(l) && (size_t)interp.get_P(l).cols() == mg.get_n_dofs(l + 1));
      CHECK(interp.get_R(l).rows() == interp.get_P(l).cols() && interp.get_R(l).nonZeros() == interp.get_P(l).nonZeros());
    }
    // R e = P^T e through the stored operators (generic device SpMV) against P's columns
    Vec r((size_t)mg.get_n_dofs(0));
    for (size_t i = 0; i < r.size(); ++i) r[i] = std::cos(0.3 * i);
    const Vec fc = interp.restriction(r, 0);
    const Mat& P = interp.get_P(0);
    double err = 0.0;
    for (int J = 0; J < P.cols(); ++J) {
      double s = 0.0;
      for (int p = P.outerIndexPtr()[J]; p < P.outerIndexPtr()[J + 1]; ++p) s += P.valuePtr()[p] * r[P.innerIndexPtr()[p]];
      err = std::fmax(err, std::fabs(s - fc[J]));
    }
    CHECK(err <= 1e-12);
    mg.solve_pcg(1e-8, 100);
    std::printf("rectangular %d x %d: %zu levels, PCG %zu iterations, relative residual %.3g\n", nx, ny, L,
                mg.iterations_done(), mg.last_error());
    CHECK(mg.last_error() <= 1e-8 && mg.iterations_done() <= 30);
  }
  std::printf("%d failed\n", g_failed);
  return g_failed == 0 ? 0 : 1;
}
