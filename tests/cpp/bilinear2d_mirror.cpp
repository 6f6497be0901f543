// C++ check of BilinearInterpolator2D in the include/amg mirror headers: the operators it builds,
// its rejection of sizes off the coarse rule, and (on the GPU) a Multigrid that picks the 2-D
// transfer from it and converges in a grid-size independent number of V-cycles.
#include <cmath>
#include <cstdio>
#include <string>
#include <stdexcept>

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
  AMG::BilinearInterpolator2D<double> bi(2);
  CHECK(bi.device_transfer() == AMGB_TRANSFER_BILINEAR_2D);
  bi.make_operators(5 * 5, 2 * 2, 0);
  const Mat& P = bi.get_P(0);
  CHECK(P.rows() == 25 && P.cols() == 4 && P.nonZeros() == 36);
  // column 0 = rows (y, x), y, x in {0, 1, 2}: weights .25 .5 .25 / .5 1 .5 / .25 .5 .25
  CHECK(P.innerIndexPtr()[0] == 0 && P.valuePtr()[0] == 0.25 && P.innerIndexPtr()[4] == 6 && P.valuePtr()[4] == 1.0);
  CHECK(bi.get_R(0).rows() == 4 && bi.get_R(0).cols() == 25);
  bool threw = false;
  try {
    bi.make_operators(5 * 5, 3 * 3, 0);
  } catch (const std::invalid_argument&) {
    threw = true;
  }
  CHECK(threw);
  if (argc > 1 && std::string(argv[1]) == "gpu") {
    const size_t m = 129, L = 5;
    Mat A = AMG::Grid<double>::laplacian(m);
    Vec b = AMG::Grid<double>::rhs(m);
    AMG::BilinearInterpolator2D<double> interp(L);
    AMG::SparseGaussSeidel<double> gs;
    AMG::Multigrid<double> mg(&interp, &gs, A, b, L, 1e-9, 1, 100);
    CHECK(mg.get_n_dofs(1) == 64 * 64 && interp.get_P(0).cols() == 64 * 64);
    CHECK(amgb_hierarchy_transfer(mg.handle()) == AMGB_TRANSFER_BILINEAR_2D);
    for (int k = 0; k < 8; ++k) mg.vcycle();
    double bb = 0.0;
    for (long i = 0; i < (long)b.size(); ++i) bb += b[i] * b[i];
    const double rel = std::sqrt(AMG::rss(A, mg.get_soln(0), b) / bb);
    std::printf("2-D hierarchy: relative residual %.3g after 8 V-cycles\n", rel);
    CHECK(rel <= 1e-8);
  }
  std::printf("%d failed\n", g_failed);
  return g_failed == 0 ? 0 : 1;
}
