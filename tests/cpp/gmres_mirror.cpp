// C++ check of Multigrid::solve_gmres in the include/amg mirror headers: it compiles against the stand-in
// types and the Eigen shim, and (on the GPU) solves upwind convection-diffusion on a 65 x 65 grid -- an
// unsymmetric matrix on which the stationary V-cycle diverges -- with a smoothed-aggregation hierarchy.
#include <cmath>
#include <cstdio>
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

// kron(T + C, I) + kron(I, T) with T = tridiag(-1, 2, -1), C = (pe / m) tridiag(-1, 1, 0): compressed CSC
static Mat convection(int m, double pe) {
  const int n = m * m;
  const double c = pe / m;
  std::vector<int> outer(n + 1, 0), inner;
  std::vector<double> val;
  for (int k = 0; k < n; ++k) {
    const int x = k % m, y = k / m;
    auto put = [&](int r, double v) {
      inner.push_back(r);
      val.push_back(v);
    };
    if (y > 0) put(k - m, -1.0);
    if (x > 0) put(k - 1, -1.0);
    put(k, 4.0 + c);
    if (x + 1 < m) put(k + 1, -1.0);
    if (y + 1 < m) put(k + m, -1.0 - c);
    outer[k + 1] = (int)inner.size();
  }
#if AMGB_HAVE_EIGEN
  return Eigen::Map<const Eigen::SparseMatrix<double>>(n, n, (int)inner.size(), outer.data(), inner.data(), val.data());
#else
  return Mat(n, n, std::move(outer), std::move(inner), std::move(val));
#endif
}

int main(int argc, char** argv) {
  if (argc > 1 && std::string(argv[1]) == "gpu") {
    const int m = 65, n = m * m;
    Mat A = convection(m, 10.0);
    Vec b(n);
    for (int i = 0; i < n; ++i) b[i] = std::sin(0.01 * i) + 0.5 * std::cos(0.37 * i);
    AMG::SmoothedAggregationInterpolator<double> interp(25);
    AMG::DampedJacobi<double> jac(2.0 / 3.0, 2);
    AMG::Multigrid<double> mg(&interp, &jac, A, b, 25, 1e-9, 1, 100);
    const Vec& x = mg.solve_gmres(1e-8, 30, 200);
    double rr = 0.0, bb = 0.0;  // the true residual, recomputed here
    for (int i = 0; i < n; ++i) {
      const int xg = i % m, yg = i / m;
      double ax = (4.0 + 10.0 / m) * x[i];
      if (yg > 0) ax += (-1.0 - 10.0 / m) * x[i - m];
      if (yg + 1 < m) ax += -1.0 * x[i + m];
      if (xg > 0) ax += -1.0 * x[i - 1];
      if (xg + 1 < m) ax += -1.0 * x[i + 1];
      rr += (b[i] - ax) * (b[i] - ax);
      bb += b[i] * b[i];
    }
    const double rel = std::sqrt(rr / bb);
    std::printf("convection %d^2: %zu levels, GMRES(30) %zu steps, relative residual %.3g (recomputed %.3g)\n", m,
                mg.get_n_levels(), mg.iterations_done(), mg.last_error(), rel);
    CHECK(mg.last_error() <= 1e-8 && rel <= 1.05e-8);
    CHECK(mg.iterations_done() >= 1 && mg.iterations_done() < 60);
    CHECK(mg.error_history().size() == mg.iterations_done());
  }
  std::printf("%d failed\n", g_failed);
  return g_failed == 0 ? 0 : 1;
}
