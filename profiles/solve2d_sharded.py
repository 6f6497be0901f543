"""The sharded bilinear 2-D V-cycle across the GPUs of one node: Poisson (Grid::laplacian, eps_y = 1)
at 4097^2 and 8193^2, BilinearInterpolator2D, damped Jacobi 2+2, fast arithmetic.  Launch once per world:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node W profiles/solve2d_sharded.py [--n 4097,8193]

World 1 builds the unsharded hierarchy (amgb_hierarchy_create); world >= 2 the line-block sharded one
with the default min_rows_per_rank (2^18).  Rank 0 prints one JSON line per grid size with:

  ms_per_vcycle      host clock over 30 amgb_vcycles (graph replays) after 5 warm-up cycles, between a
                     barrier plus stream synchronise and a stream synchronise; the slowest rank's time
  cycles, time_to_tol_s   solve_relative to ||b - A u|| / ||b|| <= 1e-8 from u = 0 (host clock between a
                     barrier and the solve's return, which ends in a stream synchronise)
  host_rel_residual  ||b - A u|| / ||b|| recomputed with scipy from get_soln(0)
  phase_times        amgb_hierarchy_phase_times over 10 un-captured cycles on rank 0, ms: sharded levels
                     down, gather of the first replicated right-hand side, the replicated levels, sharded
                     levels up
  n_sharded_levels, halo_exchanges_per_vcycle, halo_mode, and the GPU name and power limit.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT]
sys.dont_write_bytecode = True

amg = importlib.import_module("algebraic-multigrid_b200")


def gpu_info(device):
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", str(device)],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001 -- reported, not fatal
        power = "unknown (%s)" % e
    return {"gpu": torch.cuda.get_device_name(device), "power_limit": power}


def levels_2d(m):
    L = 1
    while m // 2 >= 8:  # coarsest grid 8..15 lines, as profiles/solve2d.py
        m //= 2
        L += 1
    return L


def slowest(x, world):
    if world == 1:
        return x
    t = torch.tensor([x], dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t[0])


def sync(mg, world):
    mg.synchronize()
    if world > 1:
        dist.barrier()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", default="4097,8193")
    ap.add_argument("--rel-tol", type=float, default=1e-8)
    args = ap.parse_args()
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", rank))
    if amg.device_count() < world:
        raise SystemExit("needs %d GPUs, the node has %d" % (world, amg.device_count()))
    torch.cuda.set_device(local)
    amg.lib().amgb_set_device(local)
    comm = None
    if world > 1:
        dist.init_process_group("gloo")

        def ex(raw):
            box = [raw]
            dist.broadcast_object_list(box, src=0)
            return box[0]
        comm = amg.Comm(rank, world, ex)
    info = gpu_info(local)
    for m in [int(x) for x in args.n.split(",")]:
        A, b = amg.Grid.laplacian(m), amg.Grid.rhs(m)
        L = levels_2d(m)
        t0 = time.perf_counter()
        mg = amg.Multigrid(amg.BilinearInterpolator2D(L), amg.DampedJacobi(2.0 / 3.0, 2), A, b, L, 1e-9, 1, 100,
                           comm=comm, arith=amg.ARITH_FAST)
        setup_s = slowest(time.perf_counter() - t0, world)
        mg.vcycles(5)
        sync(mg, world)
        t0 = time.perf_counter()
        mg.vcycles(30)
        mg.synchronize()
        ms = slowest((time.perf_counter() - t0) * 1e3 / 30, world)
        exchanges = mg.halo_exchanges_per_vcycle()
        phases = mg.phase_times(10)
        mg.set_soln(0, np.zeros(m * m))
        sync(mg, world)
        t0 = time.perf_counter()
        mg.solve_relative(args.rel_tol)
        solve_s = slowest(time.perf_counter() - t0, world)
        u = mg.get_soln(0)
        if rank == 0:
            rel = float(np.linalg.norm(b - A.to_scipy() @ u) / np.linalg.norm(b))
            out = {"config": "bl2d_jacobi_sharded", "n": m, "world": world, "levels": L, "arith": "fast",
                   "smoother": "jacobi 2+2", "setup_s": round(setup_s, 3), "ms_per_vcycle": round(ms, 4),
                   "cycles": mg.iters_done, "reported_rel": mg.last_error, "host_rel_residual": rel,
                   "converged": rel <= args.rel_tol, "time_to_tol_s": round(solve_s, 4),
                   "phase_times_ms": {k: round(v, 4) for k, v in phases.items()},
                   "n_sharded_levels": mg.n_sharded_levels(), "halo_exchanges_per_vcycle": exchanges,
                   "halo_mode": mg.halo_mode(), "local_range_0": mg.local_range(0)}
            out.update(info)
            print(json.dumps(out), flush=True)
        del mg, A, b, u
    if world > 1:
        dist.barrier()
        del comm
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
