"""Time-to-solution of the 4097^2 Poisson problem (--eps: eps_y of Grid::laplacian, 1e-3 for the
anisotropic bench config aniso4097) with the reference's 1-D transfer and with the bilinear 2-D
transfer (TRANSFER_BILINEAR_2D).  One JSON line per configuration on stdout:

  linear_pcg        LinearInterpolator, damped Jacobi 2+2 (fast arithmetic), solve_pcg
  linear_relative   LinearInterpolator, damped Jacobi 2+2 (fast arithmetic), solve_relative, <= 100 cycles
  bl2d_jacobi       BilinearInterpolator2D, damped Jacobi 2+2 (fast arithmetic), solve_relative
  bl2d_gs           BilinearInterpolator2D, symmetric Gauss-Seidel x1 (GS_AUTO), solve_relative
  bl2d_pcg          BilinearInterpolator2D, damped Jacobi 2+2 (fast arithmetic), solve_pcg
  bl2d_line_x       BilinearInterpolator2D, zebra X-line Gauss-Seidel x1 (fast arithmetic), solve_relative
  bl2d_line_alt     BilinearInterpolator2D, alternating zebra line Gauss-Seidel x1 (fast), solve_relative
  bl2d_line_x_pcg   BilinearInterpolator2D, zebra X-line Gauss-Seidel x1 (fast arithmetic), solve_pcg

Every solve_relative is capped at 100 V-cycles.

Each line: setup seconds (host clock around the constructor), cycles or PCG iterations, ms per V-cycle
(CUDA events over >= 20 graph replays after warm-up), time to rel_tol (host clock around the solve, which
ends in a stream synchronise), the final ||b - A u|| / ||b|| recomputed on the host with scipy from
get_soln(0), launches per V-cycle, the Gauss-Seidel kernel of every level, and for the 2-D hierarchies
the level-0 times of k_residual (kind 1), k_residual_restrict2d (kind 2) and k_prolong_add2d (kind 3)
with their algorithmic bytes (SURVEY.md section 8d with N_1 = N_0 / 4) over a device-to-device copy
bandwidth measured in the same run; for the line smoothers also one X-line and one Y-line pass of one
colour (kinds 12 and 13: k_line_rhs + k_line_solve on the N_0 / 2 rows of the colour), whose bytes are
per row f, the k off-line coefficients, the other colour's u, t written and read back as y, the three
factors and u written: 8 (9 + k) bytes.  A last line checks 3 V-cycles from zero against the 2-D oracle
(tests/oracle_bilinear2d.py) at --parity-n.  GPU name and power limit are part of every line.

    python profiles/solve2d.py [--n 4097] [--eps 1.0] [--parity-n 1025] [--rel-tol 1e-8] [--only a,b]
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
sys.dont_write_bytecode = True

amg = importlib.import_module("algebraic-multigrid_b200")


def gpu_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001 -- reported, not fatal
        power = "unknown (%s)" % e
    return {"gpu": name, "power_limit": power}


def copy_bandwidth_gbs(nbytes=1 << 30, reps=20):
    """Device-to-device copy: (read + write bytes) / time, CUDA events."""
    import torch
    x = torch.empty(nbytes // 8, dtype=torch.float64, device="cuda")
    y = torch.empty_like(x)
    for _ in range(3):
        y.copy_(x)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        y.copy_(x)
    e1.record()
    e1.synchronize()
    return 2.0 * nbytes * reps / (e0.elapsed_time(e1) * 1e-3) / 1e9


def levels_linear(n0):
    L, n = 1, n0
    while n > 200:  # bench.py's default: coarsen until <= 200 DOF
        n = amg.lib().amgb_n_H_dofs_from_n_h_dofs(n)
        L += 1
    return L


def levels_2d(m):
    L = 1
    while m // 2 >= 8:  # coarsest grid 8..15 lines (<= 225 DOF)
        m //= 2
        L += 1
    return L


def ms_per_cycle(mg, warmup=5, reps=30):
    import torch
    s = torch.cuda.Stream()
    mg.set_stream(s.cuda_stream)
    with torch.cuda.stream(s):
        for _ in range(warmup):
            mg.vcycle()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(s)
        for _ in range(reps):
            mg.vcycle()
        e1.record(s)
    e1.synchronize()
    mg.set_stream(0)
    return e0.elapsed_time(e1) / reps


def run(name, interp, smoother, solver, A, b, As, m, eps, rel_tol, bw, info, arith):
    L = levels_2d(m) if interp is amg.BilinearInterpolator2D else levels_linear(m * m)
    t0 = time.perf_counter()
    mg = amg.Multigrid(interp(L), smoother, A, b, L, 1e-9, 1, 100, arith=arith)
    setup_s = time.perf_counter() - t0
    mg.vcycle()  # graph capture and first launch outside the timed solve
    mg.synchronize()
    mg.set_soln(0, np.zeros(m * m))
    t0 = time.perf_counter()
    if solver == "pcg":
        mg.solve_pcg(rel_tol, 2000)
    else:
        mg.solve_relative(rel_tol)
    solve_s = time.perf_counter() - t0
    u = mg.get_soln(0)
    rel = float(np.linalg.norm(b - As @ u) / np.linalg.norm(b))
    out = {"config": name, "n": m, "eps_y": eps, "levels": L, "transfer": mg.transfer(), "solver": solver,
           "setup_s": round(setup_s, 3), "iters": mg.iters_done, "reported_rel": mg.last_error,
           "host_rel_residual": rel, "converged": rel <= rel_tol, "time_to_tol_s": round(solve_s, 4)}
    out["ms_per_vcycle"] = ms_per_cycle(mg)
    out["launches_per_vcycle"] = mg.launches_per_vcycle()
    out["gs_kernel"] = [mg.gs_kernel(l) for l in range(L)]
    if mg.transfer() == amg.TRANSFER_BILINEAR_2D:
        N0, N1, nnz0 = m * m, (m * m) // 4, mg.nnz_device(0)
        kern = {}
        for kind, label, nbytes in ((1, "k_residual", 12 * nnz0 + 28 * N0 + 4),
                                    (2, "k_residual_restrict2d", 12 * nnz0 + 20 * N0 + 4 + 8 * N1),
                                    (3, "k_prolong_add2d", 8 * N1 + 16 * N0)):
            ms = mg.time_kernel(0, kind, warmup=5, reps=30)
            gbs = nbytes / (ms * 1e-3) / 1e9
            kern[label] = {"ms": ms, "alg_bytes": nbytes, "GBs": gbs, "share_of_copy_bw": gbs / bw}
        if getattr(smoother, "kind", None) == amg.SMOOTHER_LINE_GS:
            k_off = int(round(nnz0 / N0)) - 3
            for kind, label in ((12, "x_pass"), (13, "y_pass")):
                nbytes = (N0 // 2) * 8 * (9 + k_off)
                ms = mg.time_kernel(0, kind, warmup=3, reps=10)
                gbs = nbytes / (ms * 1e-3) / 1e9
                kern[label] = {"ms": ms, "alg_bytes": nbytes, "GBs": gbs, "share_of_copy_bw": gbs / bw}
        out["level0_kernels"] = kern
    out.update(info)
    out["copy_bw_GBs"] = bw
    return out


def parity(n, eps):
    import oracle as O
    import oracle_bilinear2d as O2
    import oracle_linegs2d as OL
    A, b = amg.Grid.laplacian(n, eps), amg.Grid.rhs(n)
    L = levels_2d(n)
    res = {"config": "parity_3_cycles", "n": n, "eps_y": eps, "levels": L}
    for label, make, kind, iters, arith in (
            ("line_x_reference", lambda: amg.LineGaussSeidel(1, amg.LINES_X), OL.SMOOTHER_LINE_GS, 1,
             amg.ARITH_REFERENCE),
            ("line_alt_fast", lambda: amg.LineGaussSeidel(1, amg.LINES_ALTERNATING), OL.SMOOTHER_LINE_GS, 1,
             amg.ARITH_FAST),
            ("jacobi_reference", lambda: amg.DampedJacobi(2.0 / 3.0, 2), O.SMOOTHER_JACOBI, 2, amg.ARITH_REFERENCE),
            ("jacobi_fast", lambda: amg.DampedJacobi(2.0 / 3.0, 2), O.SMOOTHER_JACOBI, 2, amg.ARITH_FAST),
            ("gs_auto", lambda: amg.SparseGaussSeidel(), O.SMOOTHER_GS, 1, amg.ARITH_REFERENCE)):
        mg = amg.Multigrid(amg.BilinearInterpolator2D(L), make(), A, b, L, 1e-9, 1, 100, arith=arith)
        lines = amg.LINES_ALTERNATING if label == "line_alt_fast" else amg.LINES_X
        mo = OL.Multigrid(O.laplacian(n, eps), b, L, 1e-9, 1, 100, kind, iters, 2.0 / 3.0, lines=lines)
        for _ in range(3):
            mg.vcycle()
            mo.vcycle()
        u, uo = mg.get_soln(0), mo.u(0)
        res[label] = {"bit_identical": u.tobytes() == uo.tobytes(),
                      "rel_diff": float(np.linalg.norm(u - uo) / np.linalg.norm(uo))}
    return res


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--n", type=int, default=4097)
    p.add_argument("--parity-n", type=int, default=1025)
    p.add_argument("--rel-tol", type=float, default=1e-8)
    p.add_argument("--eps", type=float, default=1.0, help="eps_y of the operator")
    p.add_argument("--only", default="", help="comma-separated subset of the configurations")
    a = p.parse_args()
    if amg.device_count() < 1:
        raise SystemExit("needs a CUDA device")
    info = gpu_info()
    bw = copy_bandwidth_gbs()
    m = a.n
    A, b = amg.Grid.laplacian(m, a.eps), amg.Grid.rhs(m)
    As = A.to_scipy()
    J = lambda: amg.DampedJacobi(2.0 / 3.0, 2)  # noqa: E731
    configs = [
        ("linear_pcg", amg.LinearInterpolator, J, "pcg", amg.ARITH_FAST),
        ("linear_relative", amg.LinearInterpolator, J, "relative", amg.ARITH_FAST),
        ("bl2d_jacobi", amg.BilinearInterpolator2D, J, "relative", amg.ARITH_FAST),
        ("bl2d_gs", amg.BilinearInterpolator2D, lambda: amg.SparseGaussSeidel(), "relative", amg.ARITH_REFERENCE),
        ("bl2d_pcg", amg.BilinearInterpolator2D, J, "pcg", amg.ARITH_FAST),
        ("bl2d_line_x", amg.BilinearInterpolator2D, lambda: amg.LineGaussSeidel(1, amg.LINES_X), "relative",
         amg.ARITH_FAST),
        ("bl2d_line_alt", amg.BilinearInterpolator2D, lambda: amg.LineGaussSeidel(1, amg.LINES_ALTERNATING),
         "relative", amg.ARITH_FAST),
        ("bl2d_line_x_pcg", amg.BilinearInterpolator2D, lambda: amg.LineGaussSeidel(1, amg.LINES_X), "pcg",
         amg.ARITH_FAST),
    ]
    only = set(filter(None, a.only.split(",")))
    for name, interp, make, solver, arith in configs:
        if only and name not in only:
            continue
        print(json.dumps(run(name, interp, make(), solver, A, b, As, m, a.eps, a.rel_tol, bw, info, arith)), flush=True)
    if a.parity_n > 0:
        out = parity(a.parity_n, a.eps)
        out.update(info)
        print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
