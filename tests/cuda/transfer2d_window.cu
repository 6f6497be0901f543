// The windowed 2-D transfer kernels (kernels.cuh) on a sub-range of lines, addressed through
// pointers shifted to the window's first line as a rank of a sharded level addresses its block,
// against the same kernels on the whole level: the window's coarse lines (restriction) and fine
// lines (prolongation) must be bit-identical, everything outside the window untouched.
// Usage: transfer2d_window m   -> prints "OK <windows>" or the first mismatch, exit code 0 / 1.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "kernels.cuh"

using namespace amgb::dev;

#define CK(x)                                                                        \
  do {                                                                               \
    cudaError_t e_ = (x);                                                            \
    if (e_ != cudaSuccess) {                                                         \
      std::printf("CUDA error %s at line %d\n", cudaGetErrorString(e_), __LINE__);   \
      std::exit(2);                                                                  \
    }                                                                                \
  } while (0)

static double rnd(unsigned long long& s) {
  s = s * 6364136223846793005ull + 1442695040888963407ull;
  return (double)(s >> 11) / (double)(1ull << 53) - 0.5;
}

int main(int argc, char** argv) {
  const int m = argc > 1 ? std::atoi(argv[1]) : 65, mH = m / 2, n = m * m, nH = mH * mH;
  const int ld = (n + 31) / 32 * 32, offs[5] = {-m, -1, 0, 1, m};
  unsigned long long seed = 12345 + m;
  std::vector<double> val(5 * (size_t)ld, 0.0), u(n), f(n), e(nH);
  for (int r = 0; r < n; ++r) {
    const int y = r / m, x = r % m;
    const bool in[5] = {y > 0, x > 0, true, x + 1 < m, y + 1 < m};
    for (int d = 0; d < 5; ++d) val[(size_t)d * ld + r] = in[d] ? (d == 2 ? 4.0 : -1.0) + 0.1 * rnd(seed) : 0.0;
    u[r] = rnd(seed);
    f[r] = rnd(seed);
  }
  for (double& v : e) v = rnd(seed);
  double *dval, *du, *df, *de, *dfc, *duc, *dup;
  CK(cudaMalloc(&dval, val.size() * 8));
  CK(cudaMalloc(&du, n * 8));
  CK(cudaMalloc(&df, n * 8));
  CK(cudaMalloc(&de, nH * 8));
  CK(cudaMalloc(&dfc, nH * 8));
  CK(cudaMalloc(&duc, nH * 8));
  CK(cudaMalloc(&dup, n * 8));
  CK(cudaMemcpy(dval, val.data(), val.size() * 8, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(du, u.data(), n * 8, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(df, f.data(), n * 8, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(de, e.data(), nH * 8, cudaMemcpyHostToDevice));
  auto view = [&](int first_row, int rows) {
    DiaViewT<5> V;
    std::memset(&V, 0, sizeof(V));
    V.n_rows = rows;
    V.c_min = -first_row;
    V.c_max = n - 1 - first_row;
    V.ld = ld;
    V.n_diag = 5;
    for (int d = 0; d < 5; ++d) V.off[d] = offs[d];
    V.val = dval + first_row;
    return V;
  };
  const int X = (mH + kRR2X - 1) / kRR2X;
  // whole level
  std::vector<double> fc_whole(nH), up_whole(n);
  k_residual_restrict2d<DiaViewT<5>><<<dim3(X, (mH + kRR2Y - 1) / kRR2Y), 256>>>(view(0, n), du, df, m, 0, dfc, duc, mH,
                                                                             0, 0, mH);
  CK(cudaMemcpy(dup, du, n * 8, cudaMemcpyDeviceToDevice));
  k_prolong_add2d<<<dim3((m + 255) / 256, (m + 1) / 2), 256>>>(de, mH, 0, dup, m, 0, 0, m);
  CK(cudaMemcpy(fc_whole.data(), dfc, nH * 8, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(up_whole.data(), dup, n * 8, cudaMemcpyDeviceToHost));
  int windows = 0;
  for (int Y0 = 0; Y0 < mH; Y0 += 3)
    for (int Y1 : {Y0 + 1, Y0 + 2, Y0 + 9, mH}) {
      if (Y1 > mH) continue;
      const int y0 = 2 * Y0, y1 = Y1 == mH ? m : 2 * Y1;
      // restriction: fine rows [y0, min(m, 2 Y1 + 1)) lines exist in the window, nothing else
      const int fine_lines = std::min(m, 2 * Y1 + 1) - y0;
      const double nan = std::nan("");
      std::vector<double> fill(nH, nan);
      CK(cudaMemcpy(dfc, fill.data(), nH * 8, cudaMemcpyHostToDevice));
      k_residual_restrict2d<DiaViewT<5>><<<dim3(X, (Y1 - Y0 + kRR2Y - 1) / kRR2Y), 256>>>(
          view(y0 * m, fine_lines * m), du + (size_t)y0 * m, df + (size_t)y0 * m, m, y0, dfc + (size_t)Y0 * mH, nullptr,
          mH, Y0, Y0, Y1);
      std::vector<double> fc(nH);
      CK(cudaMemcpy(fc.data(), dfc, nH * 8, cudaMemcpyDeviceToHost));
      for (int J = 0; J < nH; ++J) {
        const bool inside = J / mH >= Y0 && J / mH < Y1;
        if (inside ? std::memcmp(&fc[J], &fc_whole[J], 8) != 0 : !std::isnan(fc[J])) {
          std::printf("restriction m=%d window [%d,%d) coarse row %d: %.17g vs %.17g\n", m, Y0, Y1, J, fc[J], fc_whole[J]);
          return 1;
        }
      }
      // prolongation onto fine lines [y0, y1), coarse vector addressed from line Y0 (reads line Y0 - 1 below it)
      CK(cudaMemcpy(dup, du, n * 8, cudaMemcpyDeviceToDevice));
      k_prolong_add2d<<<dim3((m + 255) / 256, (y1 - y0 + 1) / 2), 256>>>(de + (size_t)Y0 * mH, mH, Y0, dup + (size_t)y0 * m,
                                                                          m, y0, y0, y1);
      std::vector<double> up(n);
      CK(cudaMemcpy(up.data(), dup, n * 8, cudaMemcpyDeviceToHost));
      for (int k = 0; k < n; ++k) {
        const bool inside = k / m >= y0 && k / m < y1;
        if (std::memcmp(&up[k], inside ? &up_whole[k] : &u[k], 8) != 0) {
          std::printf("prolongation m=%d window [%d,%d) fine row %d: %.17g\n", m, y0, y1, k, up[k]);
          return 1;
        }
      }
      ++windows;
    }
  CK(cudaDeviceSynchronize());
  std::printf("OK %d\n", windows);
  return 0;
}
