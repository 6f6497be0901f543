// The Krylov-basis kernels of amgb_solve_gmres (csrc/krylov.cuh) against a double-double host reference:
// the multi-dot V^T w, the fused update w - V c with the dots of the reorthogonalisation, the same update
// with the sum of squares, and 0 - V y from a zero base (the solver forms t = V y with c = -y).  Every result must agree with the reference
// within a few ulps of the summed magnitudes, and a second launch on the same data must give the same
// bits.  usage: krylov_kernels N k  (prints OK on success)
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "krylov.cuh"

using namespace amgb::krylov;

#define CK(x)                                                                          \
  do {                                                                                 \
    cudaError_t e_ = (x);                                                              \
    if (e_ != cudaSuccess) {                                                           \
      std::printf("CUDA %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); \
      std::exit(2);                                                                    \
    }                                                                                  \
  } while (0)

// double-double accumulator: hi + lo carries the exact running sum to ~106 bits
struct DD {
  double hi = 0.0, lo = 0.0;
  void add(double a) {
    const double s = hi + a, bb = s - hi, err = (hi - (s - bb)) + (a - bb);
    hi = s;
    lo += err;
  }
  void add_prod(double a, double b) {
    const double p = a * b;
    add(p);
    lo += std::fma(a, b, -p);
  }
  double value() const { return hi + lo; }
};

static uint64_t g_state = 0x9E3779B97F4A7C15ull;
static double uniform() {  // [-1, 1)
  g_state = g_state * 6364136223846793005ull + 1442695040888963407ull;
  return (double)(int64_t)(g_state >> 11) / (double)(1ull << 52) - 1.0;
}

static int g_bad = 0;
static void expect_close(const char* what, int i, double got, double ref, double mag) {
  const double tol = 8.0 * 2.220446049250313e-16 * mag + 1e-300;
  if (!(std::fabs(got - ref) <= tol)) {
    if (g_bad < 10) std::printf("%s[%d]: %.17g vs reference %.17g (tolerance %.3g)\n", what, i, got, ref, tol);
    ++g_bad;
  }
}

struct Results {
  std::vector<double> h, h2, w2, ss, t;
};

int main(int argc, char** argv) {
  if (argc < 3) {
    std::printf("usage: krylov_kernels N k\n");
    return 2;
  }
  const int64_t n = std::atoll(argv[1]);
  const int k = std::atoi(argv[2]);
  const int64_t ld = basis_ld(n);
  const int nb = tiles(n);
  std::vector<double> V((size_t)(k + 1) * ld, 0.0), c(k), y(k);
  for (int i = 0; i <= k; ++i)
    for (int64_t x = 0; x < n; ++x) V[(size_t)i * ld + x] = uniform();
  for (int i = 0; i < k; ++i) c[i] = 0.5 * uniform(), y[i] = -uniform();
  const double* w = V.data() + (size_t)k * ld;  // slot k is w, as in the solver

  double *dV, *dw, *dc, *dy, *dpart, *dout, *dt;
  CK(cudaMalloc(&dV, sizeof(double) * V.size()));
  CK(cudaMalloc(&dw, sizeof(double) * ld));
  CK(cudaMalloc(&dc, sizeof(double) * k));
  CK(cudaMalloc(&dy, sizeof(double) * k));
  CK(cudaMalloc(&dpart, sizeof(double) * (size_t)k * nb));
  CK(cudaMalloc(&dout, sizeof(double) * (2 * k + 1)));
  CK(cudaMalloc(&dt, sizeof(double) * ld));
  CK(cudaMemcpy(dc, c.data(), sizeof(double) * k, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dy, y.data(), sizeof(double) * k, cudaMemcpyHostToDevice));
  // poison the padding of the basis: no kernel may read it
  CK(cudaMemset(dV, 0xff, sizeof(double) * V.size()));
  for (int i = 0; i <= k; ++i)
    CK(cudaMemcpy(dV + (size_t)i * ld, V.data() + (size_t)i * ld, sizeof(double) * n, cudaMemcpyHostToDevice));

  auto run = [&]() {
    Results R;
    R.h.resize(k), R.h2.resize(k), R.w2.resize(n), R.ss.resize(1), R.t.resize(n);
    double* dwk = dV + (size_t)k * ld;
    CK(cudaMemcpy(dw, dwk, sizeof(double) * n, cudaMemcpyDeviceToDevice));
    k_multidot<<<nb, kThreads>>>(dV, ld, k, dw, n, dpart);
    k_sum_rows<<<k, kThreads>>>(dpart, nb, dout);
    k_update<kDots><<<nb, kThreads>>>(dw, dw, dV, ld, k, dc, n, dpart);  // in place, as in the solver
    k_sum_rows<<<k, kThreads>>>(dpart, nb, dout + k);
    CK(cudaGetLastError());
    CK(cudaMemcpy(R.h.data(), dout, sizeof(double) * k, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(R.h2.data(), dout + k, sizeof(double) * k, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(R.w2.data(), dw, sizeof(double) * n, cudaMemcpyDeviceToHost));
    k_update<kSumSq><<<nb, kThreads>>>(dt, dw, dV, ld, 0, dc, n, dpart);  // k = 0: a copy and its sum of squares
    k_sum_rows<<<1, kThreads>>>(dpart, nb, dout + 2 * k);
    k_update<kNone><<<nb, kThreads>>>(dt, nullptr, dV, ld, k, dy, n, nullptr);
    CK(cudaGetLastError());
    CK(cudaMemcpy(R.ss.data(), dout + 2 * k, sizeof(double), cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(R.t.data(), dt, sizeof(double) * n, cudaMemcpyDeviceToHost));
    return R;
  };
  const Results A = run(), B = run();

  for (int i = 0; i < k; ++i) {
    const double* v = V.data() + (size_t)i * ld;
    DD dot, dot2;
    double mag = 0.0, mag2 = 0.0;
    for (int64_t x = 0; x < n; ++x) {
      dot.add_prod(v[x], w[x]);
      dot2.add_prod(v[x], A.w2[x]);
      mag += std::fabs(v[x] * w[x]);
      mag2 += std::fabs(v[x] * A.w2[x]);
    }
    expect_close("V^T w", i, A.h[i], dot.value(), mag);
    expect_close("V^T (w - V c)", i, A.h2[i], dot2.value(), mag2);
  }
  DD ss;
  double ss_mag = 0.0;
  for (int64_t x = 0; x < n; ++x) {
    DD u, t;
    double mu = std::fabs(w[x]), mt = 0.0;
    u.add(w[x]);
    for (int i = 0; i < k; ++i) {
      const double vx = V[(size_t)i * ld + x];
      u.add_prod(-c[i], vx);
      t.add_prod(-y[i], vx);
      mu += std::fabs(c[i] * vx);
      mt += std::fabs(y[i] * vx);
    }
    expect_close("w - V c", (int)x, A.w2[x], u.value(), mu);
    expect_close("0 - V y", (int)x, A.t[x], t.value(), mt);
    ss.add_prod(A.w2[x], A.w2[x]);
    ss_mag += A.w2[x] * A.w2[x];
  }
  expect_close("|w - V c|^2", 0, A.ss[0], ss.value(), ss_mag);

  auto same = [](const std::vector<double>& a, const std::vector<double>& b) {
    return a.size() == b.size() && std::memcmp(a.data(), b.data(), sizeof(double) * a.size()) == 0;
  };
  if (!(same(A.h, B.h) && same(A.h2, B.h2) && same(A.w2, B.w2) && same(A.ss, B.ss) && same(A.t, B.t))) {
    std::printf("two launches on the same data gave different bits\n");
    ++g_bad;
  }
  if (g_bad) {
    std::printf("FAILED: %d mismatches (n %lld, k %d)\n", g_bad, (long long)n, k);
    return 1;
  }
  std::printf("OK n %lld k %d blocks %d\n", (long long)n, k, nb);
  return 0;
}
