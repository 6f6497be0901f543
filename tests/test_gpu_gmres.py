"""amgb_solve_gmres on the device against tests/oracle_gmres.py: restarted GMRES right-preconditioned by one
V-cycle of smoothed-aggregation, bilinear 2-D and 1-D hierarchies, on the unsymmetric matrices of
tests/sa_matrices.py (where the stationary cycle diverges) and on symmetric ones.  The device sums its dot
products in another order than numpy, so step counts are compared to within one step; the true residual is
recomputed on the host with scipy.  Also: restarts and caps, the final state and bitwise reproducibility,
the argument and sharded-hierarchy rejections, the Krylov kernels alone (tests/cuda/krylov_kernels.cu) and
a 4097^2 convection-diffusion solve."""
import ctypes as C
import importlib
import math
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle as O
import oracle_bilinear2d as B
import oracle_sa as S
import sa_matrices as G
from oracle_gmres import gmres
from test_gpu_sa_matrices import CAP, ORACLE_SIZE, SMOOTHERS, as_amg, problem, rhs

amg = importlib.import_module("algebraic-multigrid_b200")
pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL = 1e-8


def sa_pair(name, smoother="jacobi", arith=amg.ARITH_REFERENCE):
    Ao, theta = problem(name)
    make, kind, iters = SMOOTHERS[smoother]
    b = rhs(Ao.rows)
    mg = amg.Multigrid(amg.SmoothedAggregation(CAP, theta), make(), as_amg(Ao), b, CAP, 1e-9, 1, 200, arith=arith)
    mo = S.Multigrid(Ao, b, CAP, 1e-9, 1, 200, kind, iters, 2.0 / 3.0, theta)
    return mg, mo, Ao, b


def check_against_oracle(mg, mo, Ao, b, restart=30, max_iters=200, tol=TOL):
    x = mg.solve_gmres(tol, restart, max_iters)
    it_o, rel_o, _, hist_o = gmres(Ao, b, lambda v: S.precondition(mo, v), tol, restart, max_iters)
    it = mg.iters_done
    assert abs(it - it_o) <= 1, (it, it_o)
    hist = mg.error_history()
    assert len(hist) == it
    for c in range(0, it, restart):  # within a cycle the estimate |g_{j+1}| / ||b|| never increases
        h = hist[c:c + restart]
        assert np.all(np.diff(h) <= 0.0), h
    true = np.linalg.norm(b - Ao.to_scipy() @ x) / np.linalg.norm(b)
    assert true == pytest.approx(mg.last_error, rel=1e-3, abs=1e-15)
    if rel_o <= tol:
        assert true <= 1.05 * tol, (true, it)
    return it, true


@pytest.mark.parametrize("name,smoother", [(n, "jacobi") for n in ("conv", "dir", "nine", "dirsym", "arrow", "zeros")]
                         + [("conv", "gs_auto"), ("nine", "gs_auto")])
def test_smoothed_aggregation_matches_oracle(name, smoother):
    mg, mo, Ao, b = sa_pair(name, smoother)
    check_against_oracle(mg, mo, Ao, b)


def test_fast_arithmetic():
    mg, mo, Ao, b = sa_pair("conv", arith=amg.ARITH_FAST)
    it, true = check_against_oracle(mg, mo, Ao, b)
    assert true <= 1.05 * TOL


def test_bilinear_convection():
    Ao, _ = problem("conv")
    m, L = ORACLE_SIZE["conv"], 6
    b = rhs(Ao.rows)
    mg = amg.Multigrid(amg.BilinearInterpolator2D(L), amg.DampedJacobi(2.0 / 3.0, 2), as_amg(Ao), b, L, 1e-9, 1, 200)
    mo = B.Multigrid(Ao, b, L, 1e-9, 1, 200, O.SMOOTHER_JACOBI, 2)
    it, true = check_against_oracle(mg, mo, Ao, b)
    assert it <= 11 and true <= 1.05 * TOL


def linear_pair(n, L):
    A, b = amg.Grid.laplacian(n), amg.Grid.rhs(n)
    mg = amg.Multigrid(amg.LinearInterpolator(L), amg.DampedJacobi(2.0 / 3.0, 2), A, b, L, 1e-9, 1, 200)
    mo = O.Multigrid(O.laplacian(n), b, L, 1e-9, 1, 200, O.SMOOTHER_JACOBI, 2, 2.0 / 3.0)
    return mg, mo, O.laplacian(n), b


def test_linear_transfer_poisson():
    mg, mo, Ao, b = linear_pair(35, 5)
    it, true = check_against_oracle(mg, mo, Ao, b)
    assert true <= 1.05 * TOL


@pytest.mark.parametrize("restart", [1, 5, 30])
def test_restarts(restart):
    mg, mo, Ao, b = sa_pair("nine")
    check_against_oracle(mg, mo, Ao, b, restart=restart)


def test_restart_beyond_n_exhausts_the_krylov_space():
    mg, mo, Ao, b = linear_pair(3, 2)  # 9 rows
    it, true = check_against_oracle(mg, mo, Ao, b, restart=20, tol=1e-13)
    assert it <= 9 and mg.error_history()[-1] < 1e-15 and true < 1e-13


def test_max_iters_is_reported_exactly():
    mg, mo, Ao, b = sa_pair("conv")
    mg.solve_gmres(TOL, 30, 7)
    assert mg.iters_done == 7 and len(mg.error_history()) == 7 and mg.last_error > TOL
    mg.set_soln(0, np.zeros(Ao.rows))
    mg.solve_gmres(TOL, 4, 10)  # two full cycles and two steps of a third
    assert mg.iters_done == 10 and len(mg.error_history()) == 10
    u0 = mg.get_soln(0)
    mg.solve_gmres(TOL, 30, 0)
    assert mg.iters_done == 0 and mg.get_soln(0).tobytes() == u0.tobytes()
    true = np.linalg.norm(b - Ao.to_scipy() @ u0) / np.linalg.norm(b)
    assert mg.last_error == pytest.approx(true, rel=1e-9)


def test_final_state_and_reproducibility():
    mg, mo, Ao, b = sa_pair("dir")
    u0 = np.random.default_rng(3).standard_normal(Ao.rows)
    runs = []
    for _ in range(2):
        mg.set_soln(0, u0)
        mg.set_rhs(0, b)
        x = mg.solve_gmres(TOL)
        assert mg.get_rhs(0).tobytes() == b.tobytes()
        assert mg.get_soln(0).tobytes() == x.tobytes()
        runs.append((x.tobytes(), mg.iters_done, mg.last_error, mg.error_history().tobytes()))
    assert runs[0] == runs[1]
    assert runs[0][2] <= TOL


def test_zero_rhs_returns_at_once():
    mg, mo, Ao, b = sa_pair("conv")
    u0 = np.full(Ao.rows, 0.25)
    mg.set_soln(0, u0)
    mg.set_rhs(0, np.zeros(Ao.rows))
    mg.solve_gmres(TOL)
    assert mg.iters_done == 0 and mg.last_error == 0.0 and mg.get_soln(0).tobytes() == u0.tobytes()


def test_invalid_arguments():
    mg, mo, Ao, b = sa_pair("conv")
    for args in ((-1.0, 30, 10), (math.nan, 30, 10), (TOL, 0, 10), (TOL, -3, 10), (TOL, 30, -1)):
        with pytest.raises(amg.InvalidArgument):
            mg.solve_gmres(*args)
    it, rel = C.c_int64(), C.c_double()
    assert amg.lib().amgb_solve_gmres(None, TOL, 30, 10, C.byref(it), C.byref(rel)) == amg.EINVAL
    mg.solve_gmres(TOL)  # the handle is still usable
    assert mg.last_error <= TOL


def test_sharded_hierarchy_is_rejected():
    world = 2
    if amg.device_count() < world:
        pytest.skip("needs %d GPUs" % world)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
           "--master-addr", "127.0.0.1", "--master-port", "29713", os.path.join(ROOT, "tests", "gmres_sharded_worker.py")]
    out = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert "GMRES SHARDED REJECTED OK" in out.stdout


# ---- the Krylov kernels alone, against a double-double host reference ----
@pytest.fixture(scope="module")
def krylov_exe(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("krylov") / "krylov_kernels")
    subprocess.check_call(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17",
                           "-Xcompiler", "-ffp-contract=off",
                           "-I", os.path.join(ROOT, "algebraic-multigrid_b200", "csrc"),
                           os.path.join(ROOT, "tests", "cuda", "krylov_kernels.cu"), "-o", out])
    return out


@pytest.mark.parametrize("n", [100, 100003, 4097 * 4097])
@pytest.mark.parametrize("k", [1, 31])
def test_krylov_kernels(krylov_exe, n, k):
    r = subprocess.run([krylov_exe, str(n), str(k)], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and r.stdout.startswith("OK"), r.stdout + r.stderr


# ---- scale ----
def test_convection_4097_bilinear():
    m, L = 4097, 11
    Ao = G.convection(m)
    M = Ao.to_scipy()
    b = rhs(m * m)
    mg = amg.Multigrid(amg.BilinearInterpolator2D(L), amg.DampedJacobi(2.0 / 3.0, 2), as_amg(Ao), b, L, 1e-9, 1, 1,
                       arith=amg.ARITH_FAST)
    x = mg.solve_gmres(TOL, 30, 200)
    true = np.linalg.norm(b - M @ x) / np.linalg.norm(b)
    assert mg.iters_done < 200 and true <= 1.05 * TOL, (mg.iters_done, true, mg.last_error)
