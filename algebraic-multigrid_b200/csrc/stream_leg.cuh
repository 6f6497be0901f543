// Register-streaming fused V-cycle legs for the damped-Jacobi cycle (sm_100a).
//
// One kernel per level and leg,
//   down leg: pre-smoothing sweeps -> residual -> restriction   (multigrid.hpp:268-282)
//   up leg:   coarse-grid correction -> post-smoothing sweeps    (multigrid.hpp:294-301)
// with the operator, f and the input vector read from HBM once, for the operators whose rows
// are a 3 x 3 stencil in (line, element) space: every diagonal offset is a*m + delta with
// a, delta in {-1,0,1} for a line length m (level 0 of an n x n grid: m = n, five points;
// level 1: seven points; Galerkin levels >= 2: nine points).
//
// A WARP is the unit of work: its 32 lanes are 32 consecutive rows of a line and it streams
// down a chunk of lines.  The chained stencil stages run one line behind the other in program
// order (stage s on line jj - s + 1 at step jj); every lane keeps the last three lines of each
// stage's result for its own element in registers, and the delta = -1 / +1 neighbours come from
// the adjacent lanes by warp shuffles -- no shared memory, no block barriers.  Each stage
// shrinks the correct lanes by one on both sides, so a warp owns the 32 - 2H middle lanes
// (H = stages [+ 1 for the restriction]) and neighbouring warps overlap.  The operator rows, f
// and the input of the line PF steps ahead are loaded straight into a register ring (coalesced
// 256-byte requests per warp and array: one IMAD.WIDE + one LDG each, row index clamped to the
// rows that exist instead of predicating the loads); the ring is indexed with compile-time
// slots by unrolling the line loop over its period.  The kernels use no shared memory and ask
// for the largest L1 carve-out: the halo columns neighbouring warps share are served from L1.
//
// Arithmetic (template flag FAST):
//   reference order (FAST = false): the per-row operation order of k_jacobi / k_jacobi_zero /
//     k_residual_restrict / k_prolong_add (kernels.cuh) -- separate multiply and subtract, IEEE
//     division -- i.e. the CPU oracle's: bit-identical results;
//   fast (FAST = true, amgb_options.arith = AMGB_ARITH_FAST): fused multiply-adds and
//     u + (omega / d) r with 1 / d from MUFU.RCP64H plus two Newton steps (full double accuracy up
//     to ~1 ulp).  Differences to the oracle are rounding-level (~1e-16 per operation); the
//     contract of the path is 1e-12 relative on the per-level iterates, tests/test_gpu_parity.py.
//
// Rows that do not exist (outside the level, or outside the window of a sharded level) are not
// predicated away: their loads are clamped to the nearest existing row, so they compute finite
// garbage.  No existing row reads them with a non-zero coefficient (the operator has no entry
// there), and 0 * finite = 0, so the results of the rows that are stored are unaffected.
//
// Half streaming (template flag HALF, Params::half): on a level whose operator is bitwise symmetric
// the kernel loads only the centre and upper slots 4..8 of each row.  A lower coefficient is the
// upper coefficient of the row it couples to, a(k, k+o) = a(k+o, k) for o = a*m + delta < 0, and
// that row sits on lane i + delta of the previous line (a = -1) or of the same line (slot 3): it is
// taken from registers by a shuffle when the line enters the input stage, where the ring still
// holds the previous line (one extra line is loaded before the loop for the first one).  The
// coefficient bits and the summation order do not change.  Rows k + o < 0 get an explicit 0: the
// previous line of line 0 was loaded clamped and holds row 0's non-zero upper coefficients.
//
// Multi-GPU (Params::sync.enabled): the edge warps wait for the neighbour's previous site before
// touching ghost rows and push their boundary rows into the neighbour's ghost rows at the end
// (stream_leg_api.hpp, struct Sync) -- the halo exchange costs no launch.
#pragma once
#include <cstdint>

#include <cuda_runtime.h>

#include "stream_leg_api.hpp"

namespace amgb {
namespace sleg {

__device__ __forceinline__ double rcp_refined(double d) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(d));  // MUFU.RCP64H: ~20 good bits
  double e = __fma_rn(-d, r, 1.0);
  r = __fma_rn(r, e, r);
  e = __fma_rn(-d, r, 1.0);
  return __fma_rn(r, e, r);
}

// MF: matrix-free five-point operator (Params::cst, presence of a neighbour decided from the row index)
// DICT: the operator row comes from a table of the level's distinct rows in shared memory, selected
//       by one byte per row (Params::tid / table) -- 1 instead of 8 x diagonals bytes per row from HBM
// HALF: only the centre and upper slots are loaded, the lower ones are derived (bitwise-symmetric operator)
template <int KIND, unsigned MASK, int NU, int PF_, bool FAST, bool MF = false, bool DICT = false, bool HALF = false>
struct Leg {
  static_assert(!(MF && DICT), "one operator source");
  static_assert(!MF || MASK == kMask5, "the matrix-free variant is the five-point stencil");
  static_assert(!HALF || (!MF && !DICT), "half streaming reads the DIA mirror");
  static_assert(!HALF || mirror9(MASK) == MASK, "half streaming needs slot 8 - SL for every lower slot SL");
  static constexpr int ND = popc9(MASK);
  static constexpr int NS = stages(KIND, NU);                // chained stencil stages
  static constexpr int H = lost_lanes(KIND, NU);             // lanes lost on each side
  static constexpr int PF = PF_;                             // lines in flight
  static constexpr int RS = NS + 1 + PF;                     // register-ring slots
  static constexpr int DC = popc9(MASK & 0xFu);              // rank of the centre slot (0,0)
  static constexpr int S_OUT = (KIND == UP) ? NS : NS - 1;   // stage whose result is the iterate
  static_assert((MASK >> 4) & 1u, "the diagonal must be present");
  // derived coefficients of lane 0 (delta = -1) and lane 31 (delta = +1) are garbage: those lanes
  // must be lost after the first stencil stage already
  static_assert(!HALF || H >= 1, "half streaming needs the edge lanes lost");
  static constexpr int D0 = HALF ? DC : 0;  // first operator slot loaded from memory

  struct Line {
    double a[MF ? 1 : ND];  // operator row (not loaded by the matrix-free variant)
    double f, u, e0, e1;
  };
  // per-lane constants of the matrix-free variant: the -1 / +1 neighbours exist unless the row is the
  // first / last of its grid line -- (k + base) mod m, the same for every row a lane visits
  struct Lane {
    double a_left, a_right, w;  // w = omega / diag (fast arithmetic)
    const double* table;        // DICT: the row table in shared memory
  };
  // operator row of global row kg, entries in ascending column order: -m, -1, 0, +1, +m
  static __device__ __forceinline__ void mf_row(const Params& P, const Lane& Z, int kg, double (&a)[5]) {
    a[0] = (kg >= P.m) ? P.cst[0] : 0.0;
    a[1] = Z.a_left;
    a[2] = P.cst[2];
    a[3] = Z.a_right;
    a[4] = (kg < P.n_global - P.m) ? P.cst[4] : 0.0;
  }

  // ---- arithmetic ----
  static __device__ __forceinline__ double mulsub(double acc, double a, double x) {
    if constexpr (FAST) return __fma_rn(-a, x, acc);
    else return __dsub_rn(acc, __dmul_rn(a, x));
  }
  // x + omega * (r / d); rows without a diagonal keep x (smoother semantics of kernels.cuh)
  static __device__ __forceinline__ double relax(double x, double r, double d, double omega) {
    if constexpr (FAST) {
      const double w = omega * rcp_refined(d);
      return (d == 0.0) ? x : __fma_rn(w, r, x);
    } else {
      return (d == 0.0) ? x : __dadd_rn(x, __dmul_rn(omega, __ddiv_rn(r, d)));
    }
  }
  // first sweep from the zero guess: omega * (f / d)
  static __device__ __forceinline__ double relax_zero(double f, double d, double omega) {
    if constexpr (FAST) return (d == 0.0) ? 0.0 : f * (omega * rcp_refined(d));
    else return (d == 0.0) ? 0.0 : __dmul_rn(omega, __ddiv_rn(f, d));
  }

  static __device__ __forceinline__ bool e_exists(const Params& P, int Jl) {
    return (unsigned)(Jl - P.e_lo) < (unsigned)P.e_cnt;
  }

  // the operator slots that come from memory (row index already clamped)
  static __device__ __forceinline__ void load_row(Line& L, const Params& P, int kc) {
#pragma unroll
    for (int d = D0; d < ND; ++d) L.a[d] = __ldg(P.vd[d] + kc);
  }
  // loads of the line whose row on this lane is k (clamped to the rows that exist)
  static __device__ __forceinline__ void load(Line& L, const Params& P, int k, const double* table = nullptr) {
    const int kc = min(max(k, P.row_lo), P.row_hi1);
    if constexpr (DICT) {
      const double* row = table + (int)__ldg(P.tid + kc) * ND;
#pragma unroll
      for (int d = 0; d < ND; ++d) L.a[d] = row[d];
    } else if constexpr (!MF) {
      load_row(L, P, kc);
    }
    L.f = __ldg(P.f + kc);
    if (KIND != DOWN_ZERO) L.u = __ldg(P.uin + kc);
    if (KIND == UP) {
      // (P e)[k]: odd k: 1 e[J]; even k: .5 e[J-1] + .5 e[J], J = k >> 1, terms outside
      // [0, n_coarse) absent (interpolator.hpp:118-125)
      const int Jl = ((kc + P.base) >> 1) - P.cbase;
      const int last = P.e_lo + (P.e_cnt > 0 ? P.e_cnt - 1 : 0);
      L.e1 = __ldg(P.e + min(max(Jl, P.e_lo), last));
      L.e0 = __ldg(P.e + min(max(Jl - 1, P.e_lo), last));
    }
  }

  // L2 prefetch of the operator / f / input rows of a line further ahead than the register ring:
  // no registers, the later LDG then hits L2 (lower latency = fewer lines needed in flight)
  static __device__ __forceinline__ void prefetch(const Params& P, int k) {
    const int kc = min(max(k, P.row_lo), P.row_hi1);
    if constexpr (!MF && !DICT) {
#pragma unroll
      for (int d = D0; d < ND; ++d) asm volatile("prefetch.global.L2 [%0];" ::"l"(P.vd[d] + kc));
    }
    asm volatile("prefetch.global.L2 [%0];" ::"l"(P.f + kc));
    if (KIND != DOWN_ZERO) asm volatile("prefetch.global.L2 [%0];" ::"l"(P.uin + kc));
  }

  // input value of a row (stage 0); kg = global row
  static __device__ __forceinline__ double input(const Line& L, const Params& P, int kg) {
    if (KIND == DOWN_U) return L.u;
    if (KIND == DOWN_ZERO) return relax_zero(L.f, MF ? P.cst[2] : L.a[MF ? 0 : DC], P.omega);
    const int Jl = (kg >> 1) - P.cbase;
    const bool odd = kg & 1;
    const double e1 = e_exists(P, Jl) ? L.e1 : 0.0;
    const double e0 = (!odd && e_exists(P, Jl - 1)) ? L.e0 : 0.0;
    if constexpr (FAST) {
      return odd ? L.u + e1 : __fma_rn(0.5, e0 + e1, L.u);
    } else {
      double acc = 0.0;
      if (odd) {
        acc = __dadd_rn(acc, __dmul_rn(1.0, e1));
      } else {
        acc = __dadd_rn(acc, __dmul_rn(0.5, e0));
        acc = __dadd_rn(acc, __dmul_rn(0.5, e1));
      }
      return __dadd_rn(L.u, acc);
    }
  }

  // HALF: lower slot SL of line L (global row kg on this lane) from upper slot 8 - SL of row kg + o,
  // o = a * m + delta: lane i + delta of the previous line Lp (a = -1) or of L itself (a = 0)
  template <int SL>
  static __device__ __forceinline__ void derive_slot(Line& L, const Line& Lp, int m, int kg) {
    if constexpr (SL < 4 && ((MASK >> SL) & 1u)) {
      constexpr int d = popc9(MASK & ((1u << SL) - 1u));
      constexpr int du = popc9(MASK & ((1u << (8 - SL)) - 1u));
      constexpr int a = SL / 3 - 1, dl = SL % 3 - 1;
      const double src = (a < 0) ? Lp.a[du] : L.a[du];
      double v = src;
      if constexpr (dl < 0) v = __shfl_up_sync(0xffffffffu, src, 1);
      if constexpr (dl > 0) v = __shfl_down_sync(0xffffffffu, src, 1);
      L.a[d] = (kg + a * m + dl >= 0) ? v : 0.0;  // the row before the level start was loaded clamped
    }
  }
  static __device__ __forceinline__ void derive(Line& L, const Line& Lp, int m, int kg) {
    derive_slot<0>(L, Lp, m, kg);
    derive_slot<1>(L, Lp, m, kg);
    derive_slot<2>(L, Lp, m, kg);
    derive_slot<3>(L, Lp, m, kg);
  }

  template <int SL, class Row>
  static __device__ __forceinline__ void slot(const Row& a_row, double xm, double x0, double xp, double& acc) {
    if constexpr ((MASK >> SL) & 1u) {
      constexpr int d = popc9(MASK & ((1u << SL) - 1u));
      constexpr int a = SL / 3 - 1, dl = SL % 3 - 1;
      const double xl = (a < 0) ? xm : (a == 0 ? x0 : xp);
      double xv = xl;
      if constexpr (dl < 0) xv = __shfl_up_sync(0xffffffffu, xl, 1);
      if constexpr (dl > 0) xv = __shfl_down_sync(0xffffffffu, xl, 1);
      // an absent entry is stored as 0.0 and every x is finite, so acc - 0 * x == acc: no test, no select
      acc = mulsub(acc, a_row[d], xv);
    }
  }
  // f - sum a x over the row, ascending column order
  template <class Row>
  static __device__ __forceinline__ double stencil_row(double f, const Row& a_row, double xm, double x0, double xp) {
    double acc = f;
    slot<0>(a_row, xm, x0, xp, acc);
    slot<1>(a_row, xm, x0, xp, acc);
    slot<2>(a_row, xm, x0, xp, acc);
    slot<3>(a_row, xm, x0, xp, acc);
    slot<4>(a_row, xm, x0, xp, acc);
    slot<5>(a_row, xm, x0, xp, acc);
    slot<6>(a_row, xm, x0, xp, acc);
    slot<7>(a_row, xm, x0, xp, acc);
    slot<8>(a_row, xm, x0, xp, acc);
    return acc;
  }
  static __device__ __forceinline__ double stencil(const Line& L, const Params& P, const Lane& Z, int kg, double xm,
                                                   double x0, double xp) {
    if constexpr (MF) {
      double a[5];
      mf_row(P, Z, kg, a);
      return stencil_row(L.f, a, xm, x0, xp);
    } else {
      return stencil_row(L.f, L.a, xm, x0, xp);
    }
  }

  struct State {
    Line R[RS];
    double w[NS][3];  // w[s]: results of stage s (0 = input) on its last three lines
  };
  // The three-line windows rotate with the step.  When the ring period RS is a multiple of 3 the
  // slot of a line is a compile-time function of the step's position P_ in the unrolled period
  // (newest P_ % 3) and nothing moves; otherwise the window is shifted.
  static constexpr bool kStaticWindows = (RS % 3 == 0);
  static __device__ __forceinline__ constexpr int WP(int p) { return kStaticWindows ? p % 3 : 2; }        // line j + 1
  static __device__ __forceinline__ constexpr int W0(int p) { return kStaticWindows ? (p + 2) % 3 : 1; }  // line j
  static __device__ __forceinline__ constexpr int WM(int p) { return kStaticWindows ? (p + 1) % 3 : 0; }  // line j - 1
  static __device__ __forceinline__ void push(double (&w)[3], double v, int p) {
    if (kStaticWindows) {
      w[p % 3] = v;
    } else {
      w[0] = w[1];
      w[1] = w[2];
      w[2] = v;
    }
  }

  // what a warp stores: local rows [st_lo, st_lo + st_cnt) on its owned lanes
  struct Own {
    int st_lo;
    unsigned st_cnt;
    bool lane;
    __device__ __forceinline__ bool operator()(int k) const { return lane && (unsigned)(k - st_lo) < st_cnt; }
  };

  // One step: loads of line jj + 1 + PF, input stage on line jj + 1 (ring slot P_), stage s on
  // line jj - s + 1 (slot P_ - s), restriction of the residual line.  k1 = this lane's row on line jj + 1.
  template <int P_>
  static __device__ __forceinline__ void step(State& S, const Params& P, int k1, const Own& own, const Lane& Z) {
    const int m = P.m;
    // lower slots of line jj + 1 from line jj (slot P_ - 1, still in the ring); ahead of the ring load,
    // which measured fewer spills in the reference-order nine-point legs
    if constexpr (HALF) derive(S.R[P_ % RS], S.R[(P_ + RS - 1) % RS], m, k1 + P.base);
    load(S.R[(P_ + PF) % RS], P, k1 + PF * m, Z.table);
    if (P.l2_ahead > 0) prefetch(P, k1 + (PF + P.l2_ahead) * m);
    // ---- input stage, line jj + 1
    {
      const Line& L = S.R[P_ % RS];
      const double in = input(L, P, k1 + P.base);
      push(S.w[0], in, P_);
      if (S_OUT == 0 && own(k1)) P.uout[k1] = in;
    }
#pragma unroll
    for (int s = 1; s <= NS; ++s) {
      const Line& L = S.R[(P_ - s + 2 * RS) % RS];
      const int k = k1 - s * m;
      const double acc = stencil(L, P, Z, k + P.base, S.w[s - 1][WM(P_)], S.w[s - 1][W0(P_)], S.w[s - 1][WP(P_)]);
      if (KIND != UP && s == NS) {
        // residual -> restriction: f_c[J] = (.5 r[2J] + r[2J+1]) + .5 r[2J+2]   (interpolator.hpp:64-68)
        const double rm = __shfl_up_sync(0xffffffffu, acc, 1);
        const double rp = __shfl_down_sync(0xffffffffu, acc, 1);
        const int kg = k + P.base;
        if (own(k) && (kg & 1)) {
          const int J = (kg - 1) >> 1;
          if (J < P.n_coarse) {
            if constexpr (FAST) P.fc[J - P.cbase] = __fma_rn(0.5, rm + rp, acc);
            else P.fc[J - P.cbase] = __dadd_rn(__dadd_rn(__dmul_rn(0.5, rm), acc), __dmul_rn(0.5, rp));
          }
        }
      } else {
        double out;
        if constexpr (MF && FAST) out = __fma_rn(Z.w, acc, S.w[s - 1][W0(P_)]);  // omega / diag is one constant
        else out = relax(S.w[s - 1][W0(P_)], acc, MF ? P.cst[2] : L.a[MF ? 0 : DC], P.omega);
        if (s < NS) push(S.w[s], out, P_);
        if (s == S_OUT && own(k)) P.uout[k] = out;
      }
    }
  }

  // RS consecutive steps (one period of the register ring); `left` counts the steps still to
  // do and is the same for every lane of the warp, so control flow stays convergent and the
  // shuffles need no re-convergence code.
  // VOTE: `left` differs from warp to warp (sharded levels: shorter edge chunks); the early exit then goes
  // through a warp vote so that the compiler still knows the branch is warp-uniform
  template <int P_, bool VOTE = false>
  static __device__ __forceinline__ void steps(State& S, const Params& P, int& k1, int& left, const Own& own, const Lane& Z) {
    if constexpr (P_ < RS) {
      if (VOTE ? !__any_sync(0xffffffffu, left > 0) : (left <= 0)) return;
      step<P_>(S, P, k1, own, Z);
      --left;
      k1 += P.m;
      steps<P_ + 1, VOTE>(S, P, k1, left, own, Z);
    }
  }

  // ---- multi-GPU: waits and pushes of the edge warps (struct Sync)
  // Branch-free on the warp's role and convergent for the compiler (the loop exits on warp
  // votes), so the shuffles of the line loop that follows need no re-convergence code: a warp
  // that is not at this edge polls its own epoch word, which equals the value waited for.
  static __device__ __forceinline__ void wait_side(const Sync& Y, int side, bool edge) {
    // only the edge warps load anything (predicated loads, no branch); the others fall straight through
    edge = edge && Y.wait_flag[side] != nullptr;
    const unsigned long long* flag = edge ? Y.wait_flag[side] : Y.wait_epoch[side];
    unsigned long long want = 0ull;
    if (edge) want = *Y.wait_epoch[side];
    const long long t0 = clock64();
    while (true) {
      // relaxed polling (no fence per poll) ...
      unsigned long long seen = ~0ull;
      if (edge) seen = *reinterpret_cast<const volatile unsigned long long*>(flag);
      if (__all_sync(0xffffffffu, seen >= want)) break;
      if (__any_sync(0xffffffffu, clock64() - t0 > Y.timeout_cycles)) {  // a neighbour died or stalled
        *Y.timed_out = 1;
        break;
      }
      __nanosleep(32);
    }
    // ... and ONE acquire load once the flag is up: the neighbour's pushes (released system-wide before
    // its flag store) are visible to the loads that follow
    if (edge) {
      unsigned long long seen;
      asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(seen) : "l"(flag) : "memory");
    }
  }
  // wrote: this warp stored into a neighbour's memory (only then its stores need the system-wide fence)
  static __device__ __forceinline__ void signal_side(const Sync& Y, int side, int lane, bool wrote) {
    if (wrote) __threadfence_system();
    __syncwarp();
    if (lane == 0) {
      const unsigned prev = atomicAdd(Y.done[side], 1u);
      if (prev + 1u == (unsigned)Y.expected[side]) {
        *Y.done[side] = 0u;  // the next launch of this site starts from zero (stream order)
        // the other edge warps fenced their peer stores system-wide before counting themselves done; a
        // device-scope fence here orders that observation before the (cumulative) release store below
        __threadfence();
        const unsigned long long e = *Y.epoch[side] + 1ull;
        *Y.epoch[side] = e;
        if (Y.peer_flag[side] != nullptr)
          asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(Y.peer_flag[side]), "l"(e) : "memory");
      }
    }
  }
  // push the rows / coarse entries this warp stored that a neighbour keeps as ghosts: each lane
  // re-reads what it wrote itself -- the hot loop carries no push code.  Only the few lines of the
  // chunk that intersect a push range are visited, four rows per batch so their loads overlap.
  static __device__ __forceinline__ bool push_range(const double* src, double* dst, int k_lane, int m, int lo, int hi,
                                                    const Own& own) {
    // rows k = k_lane + t * m (t >= 0) of this lane inside [lo, hi) and inside what the warp stored
    lo = max(lo, own.st_lo);
    hi = min(hi, own.st_lo + (int)own.st_cnt);
    if (!own.lane || hi <= lo) return false;
    int t0 = (lo - k_lane + m - 1) / m;
    if (lo <= k_lane) t0 = 0;
    bool wrote = false;
    for (int k = k_lane + t0 * m; k < hi; k += 4 * m) {
      double v[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) v[q] = (k + q * m < hi) ? __ldcg(src + k + q * m) : 0.0;
#pragma unroll
      for (int q = 0; q < 4; ++q)
        if (k + q * m < hi) dst[k + q * m] = v[q];
      wrote = true;
    }
    return wrote;
  }
  static __device__ __forceinline__ bool push_rows(const Params& P, int k_first, const Own& own) {
    const Sync& Y = P.sync;
    bool wrote = false;
#pragma unroll
    for (int side = 0; side < 2; ++side) {
      const Push& U = Y.push_u[side];
      if (U.dst != nullptr) wrote |= push_range(P.uout, U.dst, k_first, P.m, U.begin, U.end, own);
      if (KIND != UP) {
        const Push& F = Y.push_fc[side];
        if (F.dst != nullptr) {
          // coarse entry Jl was produced by the lane that owns fine row k = 2 (Jl + cbase) + 1 - base
          const int k_lo = 2 * (F.begin + P.cbase) + 1 - P.base, k_hi = 2 * (F.end - 1 + P.cbase) + 1 - P.base + 1;
          const int lo = max(k_lo, own.st_lo), hi = min(k_hi, own.st_lo + (int)own.st_cnt);
          if (own.lane && hi > lo) {
            int t0 = (lo <= k_first) ? 0 : (lo - k_first + P.m - 1) / P.m;
            for (int k = k_first + t0 * P.m; k < hi; k += P.m) {
              const int kg = k + P.base;
              if (!(kg & 1)) continue;
              const int Jl = ((kg - 1) >> 1) - P.cbase;
              if (Jl >= F.begin && Jl < F.end && Jl + P.cbase < P.n_coarse) {
                F.dst[Jl] = __ldcg(P.fc + Jl);
                wrote = true;
              }
            }
          }
        }
      }
    }
    return __any_sync(0xffffffffu, wrote);
  }

  static __device__ __forceinline__ void run(const Params& P, double* smem_table = nullptr) {
    const int lane = threadIdx.x & 31;
    if constexpr (DICT) {  // every block keeps its own copy of the row table
      for (int i = threadIdx.x; i < P.dict_types * ND; i += blockDim.x) smem_table[i] = __ldg(P.table + i);
      __syncthreads();
    }
    // warps past the end redo the last tile without storing anything: no thread-dependent
    // branch ahead of the shuffles
    const int warp_raw = (int)((blockIdx.x * (unsigned)blockDim.x + threadIdx.x) >> 5);
    const bool dup = warp_raw >= P.n_warps;
    const int warp = dup ? P.n_warps - 1 : warp_raw;
    const int strip = warp % P.n_strips, chunk = warp / P.n_strips;
    const int i0 = strip * P.Wu, i1 = (i0 + P.Wu < P.m) ? i0 + P.Wu : P.m;
    const int j0 = P.chunk_begin(chunk), n_mine = P.chunk_lines(chunk);
    const int j1 = (j0 + n_mine < P.n_lines) ? j0 + n_mine : P.n_lines;
    Own own;
    {
      const int lo = max(j0 * P.m, P.own_begin), hi = min(j1 * P.m, P.own_end);
      own.st_lo = lo;
      own.st_cnt = (!dup && hi > lo) ? (unsigned)(hi - lo) : 0u;
      own.lane = (lane >= H && lane < H + (i1 - i0));
    }
    const bool edge_lo = P.sync.enabled && !dup && chunk < P.sync.edge_lo_chunks;
    const bool edge_hi = P.sync.enabled && !dup && chunk >= P.sync.edge_hi_chunk0;
    const bool waits = P.sync.enabled && !(P.sync.enabled & 2);  // kernel parameter: uniform (bits 1-3: timing experiments)
    if (waits) wait_side(P.sync, 0, edge_lo);  // the lower ghost rows are the first thing a lower-edge warp loads

    State S;
#pragma unroll
    for (int s = 0; s < NS; ++s) S.w[s][0] = S.w[s][1] = S.w[s][2] = 0.0;
    const int jA = j0 - NS;
    int k1 = jA * P.m + (i0 - H) + lane;  // this lane's row on line jA
    Lane Z{};
    Z.table = smem_table;
    if constexpr (MF) {
      int pos = (i0 - H + lane + P.base) % P.m;  // position of this lane's rows in their grid line
      if (pos < 0) pos += P.m;
      Z.a_left = (pos != 0) ? P.cst[1] : 0.0;
      Z.a_right = (pos != P.m - 1) ? P.cst[3] : 0.0;
      Z.w = P.omega * rcp_refined(P.cst[2]);
    }
    // steps jA - 1 .. j0 + lines + NS - 2 (a short last chunk just runs past its end); on one GPU every
    // chunk has LJ lines and the count is a kernel parameter, i.e. uniform for the compiler
    int left = (waits ? n_mine : P.LJ) + 2 * NS;
    // The upper ghost rows are the LAST thing an upper-edge warp loads: its wait for the upper neighbour
    // is deferred to the last ring period before the loads reach them, so the neighbour's latency
    // hides behind the chunk's own work.  (Pushes into the neighbour happen after the wait either way.)
    int wait_at = left;  // value of `left` at which the upper-side wait happens (period boundaries only)
    if (waits) {
      const int ghost_line = (P.own_end - 64) / P.m - 1;  // first line whose loads may touch rows >= own_end
      const int steps_before = ghost_line - jA - PF;       // steps whose loads stay below it
      if (steps_before > 0) wait_at = left - (steps_before / RS) * RS;
      if (wait_at < 1) wait_at = left - ((left - 1) / RS) * RS;  // never later than the last period
      if (__any_sync(0xffffffffu, wait_at == left)) wait_side(P.sync, 1, edge_hi);
    }
#pragma unroll
    for (int q = 0; q < PF; ++q) load(S.R[q], P, k1 + q * P.m, Z.table);
    // the line before jA, whose upper slots give jA its lower ones (slot RS - 1 is first loaded at step NS)
    if constexpr (HALF) load_row(S.R[RS - 1], P, min(max(k1 - P.m, P.row_lo), P.row_hi1));
    if (!waits) {
      // single GPU: the plain line loop (its own copy, so the multi-GPU bookkeeping below costs it nothing);
      // its trip count is a kernel parameter, i.e. provably uniform
      int left_u = P.LJ + 2 * NS;
      while (left_u > 0) steps<0>(S, P, k1, left_u, own, Z);
    } else {
      const int first = left;
      while (__any_sync(0xffffffffu, left > 0)) {
        // (votes, so the compiler knows the branches are warp-uniform and keeps the shuffles convergent)
        if (__any_sync(0xffffffffu, left == wait_at && left != first)) wait_side(P.sync, 1, edge_hi);
        steps<0, true>(S, P, k1, left, own, Z);
      }
    }

    if (edge_lo || edge_hi) {
      const bool wrote = (P.sync.enabled & 4) ? false : push_rows(P, j0 * P.m + (i0 - H) + lane, own);
      if (!(P.sync.enabled & 8)) {
        if (edge_lo) signal_side(P.sync, 0, lane, wrote);
        if (edge_hi) signal_side(P.sync, 1, lane, wrote);
      }
    }
  }
};

template <int KIND, unsigned MASK, int NU, int PF_, bool FAST, bool HALF>
__global__ void __launch_bounds__(128, (popc9(MASK) <= 5 && PF_ == 2) ? 4 : 3)
    k_stream_leg(const __grid_constant__ Params P) {
  Leg<KIND, MASK, NU, PF_, FAST, false, false, HALF>::run(P);
}
// row-type dictionary legs (at most 256 distinct operator rows on the level)
template <int KIND, unsigned MASK, int NU, bool FAST>
__global__ void __launch_bounds__(128, (popc9(MASK) <= 5) ? 4 : 3) k_stream_leg_dict(const __grid_constant__ Params P) {
  __shared__ double table[256 * popc9(MASK)];
  Leg<KIND, MASK, NU, 2, FAST, false, true>::run(P, table);
}
// matrix-free five-point legs: no operator row in the register ring, so more lines in flight and more
// resident warps
template <int KIND, int NU, int PF_, bool FAST>
__global__ void __launch_bounds__(128, 6) k_stream_leg_mf(const __grid_constant__ Params P) {
  Leg<KIND, kMask5, NU, PF_, FAST, true>::run(P);
}

}  // namespace sleg
}  // namespace amgb
