"""CPU checks of zebra line Gauss-Seidel (SMOOTHER_LINE_GS): the oracle's line solve against scipy, the
equations a pass satisfies, line_gs.cuh compiled on the host against the oracle bit for bit, the
convergence the smoother buys on anisotropic problems, and the symmetry of its V-cycle."""
import ctypes as C
import importlib
import os
import subprocess
import tempfile

import numpy as np
import pytest
import scipy.linalg as sla

import oracle as O
import oracle_linegs2d as OL
from test_bilinear2d_host import nine_point_unsymmetric, rows_dia

amg = importlib.import_module("algebraic-multigrid_b200")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def operator(kind, m):
    if kind == "unsym9":
        return nine_point_unsymmetric(m)
    return O.laplacian(m, {"iso": 1.0, "aniso_x": 1e-3, "aniso_y": 1e3}[kind])


def n_levels(m, min_lines=4):
    L = 1
    while m // 2 >= min_lines:
        m //= 2
        L += 1
    return L


def test_constants_match_the_library():
    assert (amg.SMOOTHER_LINE_GS, amg.LINES_X, amg.LINES_Y, amg.LINES_ALTERNATING) == (
        OL.SMOOTHER_LINE_GS, OL.LINES_X, OL.LINES_Y, OL.LINES_ALTERNATING)
    assert [f for f, _ in amg.Options._fields_][-1] == "lines"
    with pytest.raises(ValueError):
        amg.LineGaussSeidel(1, lines=3)


@pytest.mark.parametrize("kind", ["iso", "aniso_x", "unsym9"])
@pytest.mark.parametrize("D", [OL.X, OL.Y])
def test_line_solve_matches_solve_banded(kind, D):
    m = 37
    Cs = OL.slots(operator(kind, m), m)
    sub, den, cp = OL.factors(Cs, m, D)
    lo = OL.lines_view(Cs[OL.SUB[D]], m, D)
    di = OL.lines_view(Cs[4], m, D)
    up = OL.lines_view(Cs[OL.SUP[D]], m, D)
    t = np.random.default_rng(1).standard_normal((m, m))
    got = OL.thomas(t, sub, den, cp)
    for line in range(m):
        ab = np.zeros((3, m))
        ab[0, 1:] = up[line, :-1]
        ab[1] = di[line]
        ab[2, :-1] = lo[line, 1:]
        want = sla.solve_banded((1, 1), ab, t[line])
        assert np.max(np.abs(got[line] - want)) <= 1e-13 * np.max(np.abs(want)), line


@pytest.mark.parametrize("kind", ["iso", "aniso_x", "aniso_y", "unsym9"])
@pytest.mark.parametrize("D", [OL.X, OL.Y])
@pytest.mark.parametrize("c", [0, 1])
def test_pass_solves_the_equations_of_its_lines(kind, D, c):
    m = 33
    A = operator(kind, m)
    Cs = OL.slots(A, m)
    rng = np.random.default_rng(2)
    f, u = rng.standard_normal(m * m), rng.standard_normal(m * m)
    OL.line_pass(Cs, OL.factors(Cs, m, D), m, D, c, f, u)
    r = O.residual(A, u, f)
    Ad = A.to_scipy().tocsr()
    scale = np.abs(f) + abs(Ad) @ np.abs(u)
    on = OL.lines_view(np.arange(m * m), m, D)[c::2].reshape(-1)
    assert np.all(np.abs(r[on]) <= 1e-12 * scale[on])
    off = OL.lines_view(np.arange(m * m), m, D)[1 - c::2].reshape(-1)
    assert np.max(np.abs(r[off]) / scale[off]) > 1e-6  # the other colour is left alone


def test_rejects_wide_couplings_and_zero_pivots():
    m = 9
    A = O.laplacian(m).to_scipy().tolil()
    A[0, 2] = -0.1  # +-2 along an X-line
    A = A.tocsc()
    A.sort_indices()
    with pytest.raises(ValueError):
        OL.slots(O.Csc.from_arrays(m * m, m * m, A.indptr, A.indices, A.data), m)
    Cs = OL.slots(O.laplacian(m), m)
    Cs[4, 3 * m + 4] = 0.0
    Cs[3, 3 * m + 4] = Cs[5, 3 * m + 4] = 0.0
    with pytest.raises(ValueError, match="row %d" % (3 * m + 4)):
        OL.factors(Cs, m, OL.X)


# ---- line_gs.cuh on the host --------------------------------------------------------------------

@pytest.fixture(scope="module")
def host():
    src = os.path.join(ROOT, "tests", "cpp", "line_gs_host.cpp")
    out = os.path.join(tempfile.mkdtemp(prefix="amgb_lgs_"), "libline_gs_host.so")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-Wall",
                           "-x", "c++", src, "-o", out])
    L = C.CDLL(out)
    pd = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")
    pi = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
    L.lgs_host_factor.restype = C.c_int
    L.lgs_host_factor.argtypes = [C.c_int] * 3 + [pi, C.c_int, pd, pd, pd, pd]
    L.lgs_host_pass.restype = C.c_int
    L.lgs_host_pass.argtypes = [C.c_int] * 4 + [pi, C.c_int] + [pd] * 7
    return L


def step_major(a):  # [line, p] -> index p * m + line
    return np.ascontiguousarray(a.T).reshape(-1)


@pytest.mark.parametrize("m", [35, 64, 65, 100, 129])
@pytest.mark.parametrize("kind", ["iso", "aniso_x", "aniso_y", "unsym9"])
def test_host_build_is_bit_identical_to_oracle(host, m, kind):
    A = operator(kind, m)
    off, ld, Dv = rows_dia(A)
    val = Dv.reshape(-1).copy()
    Cs = OL.slots(A, m)
    n = m * m
    rng = np.random.default_rng(m)
    f, u0 = rng.standard_normal(n), rng.standard_normal(n)
    for D in (OL.X, OL.Y):
        sub, den, cp = (np.zeros(n) for _ in range(3))
        assert host.lgs_host_factor(m, D, len(off), off, ld, val, sub, den, cp) == -1
        fac = OL.factors(Cs, m, D)
        for got, want in zip((sub, den, cp), fac):
            assert got.tobytes() == step_major(want).tobytes(), (D, kind)
        for c in (0, 1):
            u_h, u_o = u0.copy(), u0.copy()
            assert host.lgs_host_pass(m, D, c, len(off), off, ld, val, sub, den, cp, f, u_h, np.zeros(n)) == 0
            OL.line_pass(Cs, fac, m, D, c, f, u_o)
            assert u_h.tobytes() == u_o.tobytes(), (D, c, kind)


# ---- convergence and symmetry (oracle) ----------------------------------------------------------

def cycles_to(m, eps, smoother, iters=1, lines=OL.LINES_X, cap=8):
    A, b = O.laplacian(m, eps), O.rhs(m)
    mg = OL.Multigrid(A, b, n_levels(m), 1e-30, 1, cap, smoother, iters, 2.0 / 3.0, lines=lines)
    mg.solve_relative(1e-8)
    rel = np.linalg.norm(O.residual(A, mg.u(0), b)) / np.linalg.norm(b)
    return mg.iters_done, rel


@pytest.mark.parametrize("m", [65, 129])
@pytest.mark.parametrize("eps,lines", [(1e-3, OL.LINES_X)] + [(e, OL.LINES_ALTERNATING)
                                                             for e in (1.0, 0.1, 1e-3, 1e-6, 1e3)])
def test_line_gs_reaches_1e8_within_8_cycles(m, eps, lines):
    it, rel = cycles_to(m, eps, OL.SMOOTHER_LINE_GS, lines=lines)
    assert it <= 8 and rel <= 1e-8, (it, rel)


@pytest.mark.parametrize("m", [65, 129])
@pytest.mark.parametrize("smoother,iters", [(O.SMOOTHER_JACOBI, 2), (O.SMOOTHER_GS, 1)])
def test_point_smoothers_stall_on_the_anisotropic_problem(m, smoother, iters):
    _, rel = cycles_to(m, 1e-3, smoother, iters, cap=40)
    assert rel > 1e-8, rel


@pytest.mark.parametrize("lines", [OL.LINES_X, OL.LINES_ALTERNATING])
def test_vcycle_is_a_symmetric_operator(lines):
    m = 33
    A = O.laplacian(m, 1e-2)
    mg = OL.Multigrid(A, O.rhs(m), n_levels(m), 1e-30, 1, 1, OL.SMOOTHER_LINE_GS, 1, lines=lines)

    def apply(v):
        mg.f(0)[:] = v
        mg.reset()
        mg.vcycle()
        return mg.u(0).copy()

    rng = np.random.default_rng(3)
    x, y = rng.standard_normal(m * m), rng.standard_normal(m * m)
    a, b = x @ apply(y), y @ apply(x)
    assert abs(a - b) <= 1e-12 * max(abs(a), abs(b)), (a, b)
