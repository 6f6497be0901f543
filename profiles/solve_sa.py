"""Smoothed-aggregation hierarchies (TRANSFER_SMOOTHED_AGGREGATION) at 4097^2: one JSON line per problem
on stdout.

  iso        Grid::laplacian(n), the 5-point Poisson operator
  aniso      Grid::laplacian(n, 1e-3)
  perm       Grid::laplacian(n) renumbered by a seeded random permutation (no grid order left)
  lognormal  5-point diffusion with seeded lognormal edge coefficients (tests/oracle_sa.py)

Every hierarchy: SmoothedAggregation(25) (coarsened until <= 200 rows, or until a coarse level stops
reducing: that one is the coarsest), damped Jacobi 2+2 with fast
arithmetic, PCG preconditioned by one V-cycle to ||b - A u|| / ||b|| <= 1e-8 from u = 0 with a seeded
random right-hand side.  Each line: levels, operator complexity (sum of the levels' stored entries over
level 0's), setup seconds (host clock around the constructor: aggregation, P, Galerkin products and the
device mirrors; built on the GPU unless AMGB_HOST_SETUP=1, `device_setup` says which) with its phases
(`setup_phases`: Multigrid.setup_times(), each phase ending in a stream synchronise), ms per V-cycle (CUDA events over 30 graph replays after warm-up),
PCG iterations and seconds (host clock around solve_pcg, which ends in a stream synchronise), the final
relative residual recomputed on the host with scipy, and the level-0 times of k_residual (kind 1),
k_restrict_sa (kind 2) and k_prolong_add_sa (kind 3) with their algorithmic bytes over a device-to-device
copy bandwidth measured in the same run:
  k_restrict_sa     12 nnz(P_0) (value + column of every entry of R) + 8 N_0 (r) + 16 N_1 (f, u written)
  k_prolong_add_sa  12 nnz(P_0) + 8 N_1 (e) + 16 N_0 (u read and written)
GPU name and power limit are part of every line.

    python profiles/solve_sa.py [--n 4097] [--levels 25] [--only iso,aniso] [--rel-tol 1e-8]
"""
import argparse
import importlib
import json
import os
import sys
import time

import numpy as np
import scipy.sparse as sp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "profiles")]
sys.dont_write_bytecode = True

amg = importlib.import_module("algebraic-multigrid_b200")
from solve2d import copy_bandwidth_gbs, gpu_info, ms_per_cycle  # noqa: E402


def problem(kind, m):
    """Host scipy CSC matrix (ascending row indices) of the problem."""
    if kind in ("iso", "aniso"):
        return amg.Grid.laplacian(m, 1e-3 if kind == "aniso" else 1.0).to_scipy()
    if kind == "perm":
        L = amg.Grid.laplacian(m).to_scipy()
        perm = np.random.default_rng(0).permutation(m * m)
        M = sp.csc_matrix(L[perm][:, perm])
    else:
        import oracle_sa as S
        M = S.lognormal_diffusion(m).to_scipy()
    M.sort_indices()
    return M


def run(kind, m, levels, rel_tol, bw, info):
    M = problem(kind, m)
    A = amg.CscMatrix(m * m, m * m, M.indptr, M.indices, M.data)
    b = np.random.default_rng(11).standard_normal(m * m)
    t0 = time.perf_counter()
    mg = amg.Multigrid(amg.SmoothedAggregation(levels), amg.DampedJacobi(2.0 / 3.0, 2), A, b, levels, 1e-9, 1, 100,
                       arith=amg.ARITH_FAST)
    setup_s = time.perf_counter() - t0
    L = mg.n_levels
    mg.vcycle()  # graph capture and first launch outside the timed solve
    mg.synchronize()
    mg.set_soln(0, np.zeros(m * m))
    mg.set_rhs(0, b)
    t0 = time.perf_counter()
    mg.solve_pcg(rel_tol, 200)
    solve_s = time.perf_counter() - t0
    u = mg.get_soln(0)
    rel = float(np.linalg.norm(b - M @ u) / np.linalg.norm(b))
    nnz = [mg.nnz(l) for l in range(L)]
    out = {"config": "sa_pcg_" + kind, "n": m, "levels": L, "level_rows": [mg.get_n_dofs(l) for l in range(L)],
           "operator_complexity": sum(nnz) / nnz[0], "formats": [mg.format(l) for l in range(L)],
           "setup_s": round(setup_s, 3), "device_setup": mg.device_setup,
           "setup_phases": {k: round(v, 3) for k, v in mg.setup_times().items()}, "pcg_iters": mg.iters_done, "reported_rel": mg.last_error,
           "host_rel_residual": rel, "converged": rel <= rel_tol, "time_to_tol_s": round(solve_s, 4)}
    out["ms_per_vcycle"] = ms_per_cycle(mg)
    out["launches_per_vcycle"] = mg.launches_per_vcycle()
    N0, N1, nnz0 = m * m, mg.get_n_dofs(1), mg.nnz_device(0)
    nnzP = mg.get_transfer(0).nnz
    out["nnz_P0_per_fine_row"] = nnzP / N0
    kern = {}
    for k, label, nbytes in ((1, "k_residual", 12 * nnz0 + 28 * N0 + 4),
                             (2, "k_restrict_sa", 12 * nnzP + 8 * N0 + 16 * N1),
                             (3, "k_prolong_add_sa", 12 * nnzP + 8 * N1 + 16 * N0)):
        ms = mg.time_kernel(0, k, warmup=5, reps=30)
        gbs = nbytes / (ms * 1e-3) / 1e9
        kern[label] = {"ms": ms, "alg_bytes": nbytes, "GBs": gbs, "share_of_copy_bw": gbs / bw}
    out["level0_kernels"] = kern
    out.update(info)
    out["copy_bw_GBs"] = bw
    return out


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--n", type=int, default=4097)
    p.add_argument("--rel-tol", type=float, default=1e-8)
    p.add_argument("--levels", type=int, default=25)
    p.add_argument("--only", default="iso,aniso,perm,lognormal")
    a = p.parse_args()
    if amg.device_count() < 1:
        raise SystemExit("needs a CUDA device")
    info = gpu_info()
    bw = copy_bandwidth_gbs()
    for kind in a.only.split(","):
        print(json.dumps(run(kind, a.n, a.levels, a.rel_tol, bw, info)), flush=True)


if __name__ == "__main__":
    main()
