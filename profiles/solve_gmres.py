"""Restarted GMRES(30) preconditioned by one V-cycle (amgb_solve_gmres) on 4097^2 upwind convection-diffusion
(tests/sa_matrices.py convection, Peclet 10 and 100), with the bilinear 2-D and the smoothed-aggregation
hierarchies, damped Jacobi 2+2, fast arithmetic, from u = 0 with the seeded right-hand side of the tests, to
||b - A u|| / ||b|| <= 1e-8.  One JSON line per run, on stdout and appended to solve_gmres_4097.jsonl next to
this script:

  setup_s          host clock around the constructor
  steps, solve_s   Arnoldi steps and host clock around solve_gmres (which ends in a stream synchronise)
  host_rel         the true relative residual recomputed with scipy
  ms_per_vcycle    CUDA events over 30 graph replays after warm-up
  ms_per_step_outside_vcycle   (solve_s - V-cycles * ms_per_vcycle) / steps, V-cycles = steps + GMRES cycles
  krylov_kernels   device time of k_multidot, k_update<kDots> and k_update<kSumSq> summed over one solve
                   (torch.profiler, a separate solve), with the bytes they must move over that time, against a
                   device-to-device copy measured in the same run.  Step j (k = j + 1 basis vectors of N
                   doubles) moves 8 N (k + 1) in the multi-dot, 8 N (2k + 2) in the update with the
                   reorthogonalisation dots and 8 N (k + 2) in the update with |w|^2.
GPU name and power limit are part of every line.

    python profiles/solve_gmres.py [--n 4097] [--only bilinear,sa] [--pe 10,100]
"""
import argparse
import importlib
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "profiles")]
sys.dont_write_bytecode = True

amg = importlib.import_module("algebraic-multigrid_b200")
from solve2d import copy_bandwidth_gbs, gpu_info, ms_per_cycle  # noqa: E402

RESTART, TOL, MAX_ITERS = 30, 1e-8, 200
KERNELS = {"k_multidot": lambda N, k: 8 * N * (k + 1),
           "k_update<1>": lambda N, k: 8 * N * (2 * k + 2),
           "k_update<2>": lambda N, k: 8 * N * (k + 2)}


def step_sizes(steps):
    """k of every Arnoldi step: cycles of RESTART steps, the last one shorter."""
    return [j % RESTART + 1 for j in range(steps)]


def kernel_times(mg, b, N):
    from torch.profiler import ProfilerActivity, profile
    mg.set_soln(0, np.zeros(N))
    mg.set_rhs(0, b)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        mg.solve_gmres(TOL, RESTART, MAX_ITERS)
    us = {name: 0.0 for name in KERNELS}
    for ev in prof.key_averages():
        for name in KERNELS:
            if name in ev.key:
                us[name] += ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
    return us, mg.iters_done


def run(kind, pe, m, bw, info):
    import sa_matrices as G
    Ao = G.convection(m, pe)
    N = m * m
    A = amg.CscMatrix(N, N, *Ao.arrays())
    M = Ao.to_scipy()
    b = np.random.default_rng(N).standard_normal(N)
    L = int(np.log2(m + 1)) - 1
    interp = amg.BilinearInterpolator2D(L) if kind == "bilinear" else amg.SmoothedAggregation(25)
    t0 = time.perf_counter()
    mg = amg.Multigrid(interp, amg.DampedJacobi(2.0 / 3.0, 2), A, b, 25 if kind == "sa" else L, 1e-9, 1, 1,
                       arith=amg.ARITH_FAST)
    setup_s = time.perf_counter() - t0
    mg.vcycle()  # graph capture and first launch outside the timed solve
    mg.synchronize()
    mg.set_soln(0, np.zeros(N))
    mg.set_rhs(0, b)
    mg.solve_gmres(TOL, RESTART, 2)  # allocations and first launches of the Krylov kernels
    mg.set_soln(0, np.zeros(N))
    mg.set_rhs(0, b)
    t0 = time.perf_counter()
    x = mg.solve_gmres(TOL, RESTART, MAX_ITERS)
    solve_s = time.perf_counter() - t0
    steps, reported = mg.iters_done, mg.last_error
    host_rel = float(np.linalg.norm(b - M @ x) / np.linalg.norm(b))
    ms_v = ms_per_cycle(mg)
    cycles = -(-steps // RESTART)
    vcycles = steps + cycles
    out = {"config": "gmres_%s_pe%g" % (kind, pe), "n": m, "levels": mg.n_levels, "restart": RESTART,
           "setup_s": round(setup_s, 3), "steps": steps, "gmres_cycles": cycles, "reported_rel": reported,
           "host_rel": host_rel, "converged": host_rel <= TOL, "solve_s": round(solve_s, 4),
           "ms_per_vcycle": ms_v, "vcycles": vcycles,
           "ms_per_step_outside_vcycle": (solve_s * 1e3 - vcycles * ms_v) / max(1, steps)}
    us, steps2 = kernel_times(mg, b, N)
    ks = step_sizes(steps2)
    kern = {}
    for name, nbytes in KERNELS.items():
        total = sum(nbytes(N, k) for k in ks)
        gbs = total / (us[name] * 1e-6) / 1e9 if us[name] > 0 else None
        kern[name] = {"ms_total": us[name] * 1e-3, "alg_bytes": total, "GBs": gbs,
                      "share_of_copy_bw": gbs / bw if gbs else None}
    out["krylov_kernels"] = kern
    out.update(info)
    out["copy_bw_GBs"] = bw
    return out


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--n", type=int, default=4097)
    p.add_argument("--only", default="bilinear,sa")
    p.add_argument("--pe", default="10,100")
    p.add_argument("--out", default=os.path.join(os.path.dirname(os.path.abspath(__file__)), "solve_gmres_4097.jsonl"))
    a = p.parse_args()
    if amg.device_count() < 1:
        raise SystemExit("needs a CUDA device")
    info = gpu_info()
    bw = copy_bandwidth_gbs()
    for kind in a.only.split(","):
        for pe in (float(v) for v in a.pe.split(",")):
            line = json.dumps(run(kind, pe, a.n, bw, info))
            print(line, flush=True)
            with open(a.out, "a") as f:
                f.write(line + "\n")


if __name__ == "__main__":
    main()
