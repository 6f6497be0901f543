// Instantiations and host-side dispatch of the register-streaming fused V-cycle legs
// (stream_leg.cuh).  Its own translation unit so that it compiles beside amgb.cu.
#include <algorithm>
#include <cstdlib>
#include <stdexcept>
#include <string>

#include "stream_leg.cuh"

namespace amgb {
namespace sleg {
namespace {

void check(cudaError_t e, const char* what) {
  if (e != cudaSuccess) throw std::runtime_error(std::string(what) + ": " + cudaGetErrorString(e));
}

int env_int(const char* name, int dflt) {
  const char* v = std::getenv(name);
  return v ? std::atoi(v) : dflt;
}

template <int KIND, unsigned MASK, int NU, int PF, bool FAST, bool HALF>
bool act(const Params& P, cudaStream_t s, int action, int* warps_per_sm) {
  auto kern = k_stream_leg<KIND, MASK, NU, PF, FAST, HALF>;
  if (action == 1) {
    kern<<<(P.n_warps + 3) / 4, 128, 0, s>>>(P);
    check(cudaGetLastError(), "k_stream_leg launch");
  } else if (action == 2) {
    cudaFuncAttributes fa{};
    check(cudaFuncGetAttributes(&fa, kern), "cudaFuncGetAttributes(k_stream_leg)");
    if (warps_per_sm) *warps_per_sm = std::max(1, 65536 / (std::max(fa.numRegs, 1) * 128)) * 4;
    // no shared memory: leave the whole array to the L1 (neighbouring warps' halo columns hit there)
    check(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxL1),
          "cudaFuncSetAttribute(k_stream_leg)");
  }
  return true;
}

template <int KIND, int NU, int PF, bool FAST>
bool act_mf(const Params& P, cudaStream_t s, int action, int* warps_per_sm) {
  auto kern = k_stream_leg_mf<KIND, NU, PF, FAST>;
  if (action == 1) {
    kern<<<(P.n_warps + 3) / 4, 128, 0, s>>>(P);
    check(cudaGetLastError(), "k_stream_leg_mf launch");
  } else if (action == 2) {
    cudaFuncAttributes fa{};
    check(cudaFuncGetAttributes(&fa, kern), "cudaFuncGetAttributes(k_stream_leg_mf)");
    if (warps_per_sm) *warps_per_sm = std::min(48, std::max(1, 65536 / (std::max(fa.numRegs, 1) * 128)) * 4);
    check(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxL1),
          "cudaFuncSetAttribute(k_stream_leg_mf)");
  }
  return true;
}

template <int KIND, unsigned MASK, int NU, bool FAST>
bool act_dict(const Params& P, cudaStream_t s, int action, int* warps_per_sm) {
  auto kern = k_stream_leg_dict<KIND, MASK, NU, FAST>;
  if (action == 1) {
    kern<<<(P.n_warps + 3) / 4, 128, 0, s>>>(P);
    check(cudaGetLastError(), "k_stream_leg_dict launch");
  } else if (action == 2) {
    cudaFuncAttributes fa{};
    check(cudaFuncGetAttributes(&fa, kern), "cudaFuncGetAttributes(k_stream_leg_dict)");
    if (warps_per_sm) *warps_per_sm = std::max(1, 65536 / (std::max(fa.numRegs, 1) * 128)) * 4;
  }
  return true;
}

template <int KIND, unsigned MASK, bool FAST, bool HALF>
bool by_pf(const Params& P, cudaStream_t s, int action, int* wps) {
  if (P.nu == 1) return act<KIND, MASK, 1, 2, FAST, HALF>(P, s, action, wps);
  if (P.nu != 2) return false;
  // five-point up leg: three lines in flight at 12 warps/SM measured 6 % faster than two at 16
  // (reference-order arithmetic, profiles/r1_stream_legs.md); AMGB_SLEG_PF overrides
  if constexpr (MASK == kMask5) {
    if (env_int("AMGB_SLEG_PF", (KIND == UP && !FAST) ? 3 : 2) == 3) return act<KIND, MASK, 2, 3, FAST, HALF>(P, s, action, wps);
  }
  return act<KIND, MASK, 2, 2, FAST, HALF>(P, s, action, wps);
}

template <int KIND, unsigned MASK, bool FAST>
bool by_nu(const Params& P, cudaStream_t s, int action, int* wps) {
  if (P.dict_types > 0) {
    if (P.nu == 1) return act_dict<KIND, MASK, 1, FAST>(P, s, action, wps);
    if (P.nu == 2) return act_dict<KIND, MASK, 2, FAST>(P, s, action, wps);
    return false;
  }
  if constexpr (MASK == kMask5) {
    if (P.matrix_free) {
      const int pf = env_int("AMGB_SLEG_MF_PF", 4);
      if (P.nu == 1) return pf == 2 ? act_mf<KIND, 1, 2, FAST>(P, s, action, wps) : act_mf<KIND, 1, 4, FAST>(P, s, action, wps);
      if (P.nu == 2) return pf == 2 ? act_mf<KIND, 2, 2, FAST>(P, s, action, wps) : act_mf<KIND, 2, 4, FAST>(P, s, action, wps);
      return false;
    }
  }
  return P.half ? by_pf<KIND, MASK, FAST, true>(P, s, action, wps) : by_pf<KIND, MASK, FAST, false>(P, s, action, wps);
}

template <int KIND, bool FAST>
bool by_mask(unsigned mask, const Params& P, cudaStream_t s, int action, int* wps) {
  switch (mask) {
    case kMask5: return by_nu<KIND, kMask5, FAST>(P, s, action, wps);
    case kMask7a: return by_nu<KIND, kMask7a, FAST>(P, s, action, wps);
    case kMask7b: return by_nu<KIND, kMask7b, FAST>(P, s, action, wps);
    case kMask9: return by_nu<KIND, kMask9, FAST>(P, s, action, wps);
    default: return false;
  }
}

template <bool FAST>
bool by_kind(int kind, unsigned mask, const Params& P, cudaStream_t s, int action, int* wps) {
  switch (kind) {
    case DOWN_U: return by_mask<DOWN_U, FAST>(mask, P, s, action, wps);
    case DOWN_ZERO: return by_mask<DOWN_ZERO, FAST>(mask, P, s, action, wps);
    default: return by_mask<UP, FAST>(mask, P, s, action, wps);
  }
}

}  // namespace

bool dispatch(int kind, unsigned mask, const Params& P, cudaStream_t s, int action, int* warps_per_sm, bool fast) {
  return fast ? by_kind<true>(kind, mask, P, s, action, warps_per_sm)
              : by_kind<false>(kind, mask, P, s, action, warps_per_sm);
}

}  // namespace sleg
}  // namespace amgb
