// TEST INFRASTRUCTURE ONLY -- never linked into libamgb.so.
// Host build of the smoothed-aggregation setup of algebraic-multigrid_b200/csrc/host_setup.cpp (the
// hierarchy amgb_hierarchy_create builds for AMGB_TRANSFER_SMOOTHED_AGGREGATION) for
// tests/test_sa_host.py: sa_host_build runs sa_hierarchy once, the accessors copy its levels out.
#include <cstring>
#include <stdexcept>
#include <string>

#include "../../algebraic-multigrid_b200/csrc/host_setup.hpp"

namespace {
std::vector<amgb::Csc> g_mats, g_P;
std::string g_err;
}  // namespace

extern "C" {

// 0 on success, 1 on std::invalid_argument (message in sa_host_error)
int sa_host_build(int n, const int* colptr, const int* rowidx, const double* val, double theta, int n_levels) {
  try {
    amgb::sa_hierarchy(amgb::csc_from_arrays(n, n, colptr, rowidx, val), theta, n_levels, g_mats, g_P);
    return 0;
  } catch (const std::invalid_argument& e) {
    g_err = e.what();
    return 1;
  }
}
const char* sa_host_error() { return g_err.c_str(); }
int sa_host_n_levels() { return (int)g_mats.size(); }
// kind 0: A_level, kind 1: P_level
static const amgb::Csc& pick(int kind, int level) { return kind == 0 ? g_mats[level] : g_P[level]; }
int sa_host_rows(int kind, int level) { return pick(kind, level).rows; }
int sa_host_cols(int kind, int level) { return pick(kind, level).cols; }
long long sa_host_nnz(int kind, int level) { return pick(kind, level).nnz(); }
void sa_host_copy(int kind, int level, int* colptr, int* rowidx, double* val) {
  const amgb::Csc& M = pick(kind, level);
  std::memcpy(colptr, M.colptr.data(), M.colptr.size() * sizeof(int));
  std::memcpy(rowidx, M.rowidx.data(), M.rowidx.size() * sizeof(int));
  std::memcpy(val, M.val.data(), M.val.size() * sizeof(double));
}
}
