// C++ check of LineGaussSeidel in the include/amg mirror headers: its device kind and line setting, its
// rejection of an unknown setting, and (on the GPU) a Multigrid with BilinearInterpolator2D that picks
// it up and solves an anisotropic problem in a few V-cycles.
#include <cmath>
#include <cstdio>
#include <stdexcept>
#include <string>

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

int main(int argc, char** argv) {
  AMG::LineGaussSeidel<double> lx;
  CHECK(lx.device_kind() == AMGB_SMOOTHER_LINE_GS && lx.device_lines() == AMGB_LINES_X && lx.n_iters == 1);
  AMG::LineGaussSeidel<double> la(2, AMGB_LINES_ALTERNATING);
  CHECK(la.device_lines() == AMGB_LINES_ALTERNATING && la.n_iters == 2);
  AMG::SparseGaussSeidel<double> gs;
  CHECK(gs.device_lines() == AMGB_LINES_X);
  bool threw = false;
  try {
    AMG::LineGaussSeidel<double> bad(1, 5);
  } catch (const std::invalid_argument&) {
    threw = true;
  }
  CHECK(threw);
  if (argc > 1 && std::string(argv[1]) == "gpu") {
    const size_t m = 129, L = 5;
    Mat A = AMG::Grid<double>::laplacian(m, 1e-3);
    Vec b = AMG::Grid<double>::rhs(m);
    AMG::BilinearInterpolator2D<double> interp(L);
    AMG::Multigrid<double> mg(&interp, &lx, A, b, L, 1e-9, 1, 100);
    for (int k = 0; k < 8; ++k) mg.vcycle();
    double bb = 0.0;
    for (long i = 0; i < (long)b.size(); ++i) bb += b[i] * b[i];
    const double rel = std::sqrt(AMG::rss(A, mg.get_soln(0), b) / bb);
    std::printf("eps_y = 1e-3, X-lines: relative residual %.3g after 8 V-cycles\n", rel);
    CHECK(rel <= 1e-8);
    // the stand-alone smoother (SmootherBase::smooth) moves u towards the solution
    Vec u = b;
    u.setZero();
    la.smooth(A, u, b);
    CHECK(AMG::rss(A, u, b) < bb);
  }
  std::printf("%d failed\n", g_failed);
  return g_failed == 0 ? 0 : 1;
}
