// TEST INFRASTRUCTURE ONLY -- never linked into libamgb.so.
// The host sparse product of algebraic-multigrid_b200/csrc/host_setup.cpp (multiply, the Galerkin product of
// every host-built hierarchy) for tests/test_gpu_sa_device_setup.py, which compares amgb_csc_multiply with it
// byte for byte: multiply_host computes C = L R and returns nnz(C) (-1 on an exception, message in
// multiply_host_error), multiply_host_copy copies C out.
#include <cstring>
#include <stdexcept>
#include <string>

#include "../../algebraic-multigrid_b200/csrc/host_setup.hpp"

namespace {
amgb::Csc g_C;
std::string g_err;
}  // namespace

extern "C" {

long long multiply_host(int m, int k, const int* L_colptr, const int* L_rowidx, const double* L_val, int n,
                        const int* R_colptr, const int* R_rowidx, const double* R_val) {
  try {
    g_C = amgb::multiply(amgb::csc_from_arrays(m, k, L_colptr, L_rowidx, L_val),
                         amgb::csc_from_arrays(k, n, R_colptr, R_rowidx, R_val));
    return g_C.nnz();
  } catch (const std::exception& e) {
    g_err = e.what();
    return -1;
  }
}
const char* multiply_host_error() { return g_err.c_str(); }
void multiply_host_copy(int* colptr, int* rowidx, double* val) {
  std::memcpy(colptr, g_C.colptr.data(), g_C.colptr.size() * sizeof(int));
  std::memcpy(rowidx, g_C.rowidx.data(), g_C.rowidx.size() * sizeof(int));
  std::memcpy(val, g_C.val.data(), g_C.val.size() * sizeof(double));
}
}
