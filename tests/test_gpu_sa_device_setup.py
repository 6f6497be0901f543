"""Device-side setup of smoothed-aggregation hierarchies (setup_sa.cuh) against the host setup that
AMGB_HOST_SETUP=1 selects: every level operator and prolongator byte for byte (explicit zeros and signed
zeros included), level count, formats, device entry counts and the iterates of two V-cycles, on sizes the
numpy oracle is too slow for; amgb_csc_multiply against host_setup.cpp's multiply on adversarial inputs;
the errors and the stop rule; the setup phase times."""
import ctypes as C
import importlib
import os
import subprocess
import tempfile

import numpy as np
import pytest
import scipy.sparse as sp

import oracle_sa as S

amg = importlib.import_module("algebraic-multigrid_b200")
pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "algebraic-multigrid_b200", "csrc")
CAP = 25

SMOOTHERS = {
    "jacobi": lambda: amg.DampedJacobi(2.0 / 3.0, 2),
    "color_gs": lambda: amg.MulticolorGaussSeidel(1),
    "gs_auto": lambda: amg.SparseGaussSeidel(mode=amg.GS_AUTO),
}


def from_oracle(Ao):
    return amg.CscMatrix(Ao.rows, Ao.cols, *Ao.arrays())


PROBLEMS = {
    "iso1025": lambda: amg.Grid.laplacian(1025),
    "eps1e-3_513": lambda: amg.Grid.laplacian(513, 1e-3),  # dense coarse levels: wide product columns
    "perm257": lambda: from_oracle(S.permuted_laplacian(257)[0]),
    "lognormal257": lambda: from_oracle(S.lognormal_diffusion(257)),
    "rect300x97": lambda: from_oracle(S.rectangular_poisson(300, 97)),
}


def build(A, smoother, monkeypatch, host, theta=0.08):
    if host:
        monkeypatch.setenv("AMGB_HOST_SETUP", "1")
    else:
        monkeypatch.delenv("AMGB_HOST_SETUP", raising=False)
    b = np.random.default_rng(A.rows).standard_normal(A.rows)
    try:
        return amg.Multigrid(amg.SmoothedAggregation(CAP, theta), SMOOTHERS[smoother](), A, b, CAP, 1e-9, 10, 100)
    finally:
        monkeypatch.delenv("AMGB_HOST_SETUP", raising=False)


def same_csc(M, N):
    return (M.rows == N.rows and M.cols == N.cols and M.colptr.tobytes() == N.colptr.tobytes()
            and M.rowidx.tobytes() == N.rowidx.tobytes() and M.val.tobytes() == N.val.tobytes())


@pytest.mark.parametrize("smoother", sorted(SMOOTHERS))
def test_device_setup_flag(smoother, monkeypatch):
    A = amg.Grid.laplacian(65)
    assert build(A, smoother, monkeypatch, host=False).device_setup
    assert not build(A, smoother, monkeypatch, host=True).device_setup


CASES = [(name, "jacobi") for name in sorted(PROBLEMS)] + [
    ("perm257", "color_gs"), ("rect300x97", "color_gs"), ("lognormal257", "gs_auto")]


@pytest.mark.parametrize("name,smoother", CASES)
def test_levels_and_vcycles_match_host_setup(name, smoother, monkeypatch):
    A = PROBLEMS[name]()
    dev = build(A, smoother, monkeypatch, host=False)
    ref = build(A, smoother, monkeypatch, host=True)
    assert dev.device_setup and not ref.device_setup
    L = dev.n_levels
    assert L == ref.n_levels >= 2
    for l in range(L):
        assert dev.get_n_dofs(l) == ref.get_n_dofs(l), l
        assert dev.format(l) == ref.format(l), l
        assert dev.nnz(l) == ref.nnz(l) and dev.nnz_device(l) == ref.nnz_device(l), l
        assert same_csc(dev.get_coefficient_matrix(l), ref.get_coefficient_matrix(l)), ("A", l)
    for l in range(L - 1):
        assert same_csc(dev.get_transfer(l), ref.get_transfer(l)), ("P", l)
    assert dev.vcycle_bytes() == ref.vcycle_bytes()
    for _ in range(2):
        dev.vcycle()
        ref.vcycle()
        for l in range(L):
            assert dev.get_rhs(l).tobytes() == ref.get_rhs(l).tobytes(), ("f", l)
            assert dev.get_soln(l).tobytes() == ref.get_soln(l).tobytes(), ("u", l)


# ---- amgb_csc_multiply against host_setup.cpp's multiply ----
_host = None


def host():
    """tests/cpp/multiply_host.cpp + host_setup.cpp, built into a temporary directory."""
    global _host
    if _host is None:
        so = os.path.join(tempfile.mkdtemp(prefix="amgb_multiply_host_"), "libmultiply_host.so")
        subprocess.check_call(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-Wall",
                               os.path.join(ROOT, "tests", "cpp", "multiply_host.cpp"),
                               os.path.join(CSRC, "host_setup.cpp"), "-o", so])
        L = C.CDLL(so)
        pd = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")
        pi = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
        L.multiply_host.argtypes = [C.c_int, C.c_int, pi, pi, pd, C.c_int, pi, pi, pd]
        L.multiply_host.restype = C.c_longlong
        L.multiply_host_error.restype = C.c_char_p
        L.multiply_host_copy.argtypes = [pi, pi, pd]
        _host = L
    return _host


def host_multiply(A, B):
    H = host()
    nnz = H.multiply_host(A.rows, A.cols, A.colptr, A.rowidx, A.val, B.cols, B.colptr, B.rowidx, B.val)
    assert nnz >= 0, H.multiply_host_error()
    colptr, rowidx, val = np.empty(B.cols + 1, np.int32), np.empty(nnz, np.int32), np.empty(nnz)
    H.multiply_host_copy(colptr, rowidx, val)
    return amg.CscMatrix(A.rows, B.cols, colptr, rowidx, val)


def adversarial(rows, cols, density, rng, empty_cols=0.2):
    """Random CSC with explicit +0 and -0 entries, values that cancel exactly, and empty columns."""
    M = sp.random(rows, cols, density=density, format="csc", random_state=rng)
    M.sort_indices()
    v = M.data
    k = rng.random(v.size)
    v[k < 0.1] = 0.0
    v[(k >= 0.1) & (k < 0.2)] = -0.0
    v[(k >= 0.2) & (k < 0.5)] = rng.choice([-1.0, 1.0, 0.5, -2.0], size=int(((k >= 0.2) & (k < 0.5)).sum()))
    v[k >= 0.5] = rng.standard_normal(int((k >= 0.5).sum()))
    drop = rng.random(cols) < empty_cols
    keep = np.repeat(~drop, np.diff(M.indptr))
    counts = np.where(drop, 0, np.diff(M.indptr))
    return amg.CscMatrix(rows, cols, np.concatenate([[0], np.cumsum(counts)]), M.indices[keep], v[keep])


@pytest.mark.parametrize("seed", range(6))
def test_csc_multiply_matches_host_product(seed):
    rng = np.random.default_rng(seed)
    m, k, n = (int(x) for x in rng.integers(1, 400, size=3))
    density = [0.3, 0.05, 0.01][seed % 3]
    A, B = adversarial(m, k, density, rng), adversarial(k, n, density, rng)
    C = amg.csc_multiply(A, B)
    assert same_csc(C, host_multiply(A, B))


def test_csc_multiply_negative_zero_first_term():
    # column 0 of C: one term -0.0 * 1 (stays -0.0); column 1: -0.0 + +0.0 = +0.0; column 2: (+1) + (-1) = +0
    A = amg.CscMatrix(1, 2, [0, 1, 2], [0, 0], [-0.0, 0.0])
    B = amg.CscMatrix(2, 3, [0, 1, 3, 5], [0, 0, 1, 0, 1], [1.0, 1.0, 1.0, 1.0, 1.0])
    A2 = amg.CscMatrix(1, 2, [0, 1, 2], [0, 0], [1.0, -1.0])
    C = amg.csc_multiply(A, B)
    assert same_csc(C, host_multiply(A, B)) and np.signbit(C.val[0]) and not np.signbit(C.val[1])
    C2 = amg.csc_multiply(A2, B)
    assert same_csc(C2, host_multiply(A2, B)) and C2.val[2] == 0.0 and not np.signbit(C2.val[2])


def test_csc_multiply_wide_column_uses_global_tables():
    """Lower arrowhead: dense column 0 plus the diagonal; column 0 of A A has every row (> 100,000 entries)."""
    n = 120_000
    rng = np.random.default_rng(1)
    rows = np.concatenate([np.arange(n), np.arange(1, n)])
    cols = np.concatenate([np.zeros(n, np.int64), np.arange(1, n)])
    vals = np.concatenate([rng.standard_normal(n), rng.standard_normal(n - 1)])
    M = sp.csc_matrix((vals, (rows, cols)), shape=(n, n))
    M.sort_indices()
    A = amg.CscMatrix(n, n, M.indptr, M.indices, M.data)
    C = amg.csc_multiply(A, A)
    assert C.colptr[1] - C.colptr[0] == n
    assert same_csc(C, host_multiply(A, A))


def test_csc_multiply_rejects_mismatched_shapes():
    A = amg.CscMatrix(2, 3, [0, 0, 0, 0], [], [])
    with pytest.raises(ValueError, match="inner dimensions"):
        amg.csc_multiply(A, A)


# ---- errors, stop rule, phase times ----
def error_of(A, monkeypatch, host, theta=0.08):
    with pytest.raises(ValueError) as e:
        build(A, "jacobi", monkeypatch, host, theta)
    return str(e.value)


def test_errors_match_host_setup(monkeypatch):
    L = amg.Grid.laplacian(20).to_scipy().tolil()
    L[37, 37] = 0.0
    L[250, 250] = 0.0
    Z = sp.csc_matrix(L)
    Z.sort_indices()
    Zm = amg.CscMatrix(400, 400, Z.indptr, Z.indices, Z.data)
    msg = error_of(Zm, monkeypatch, host=False)
    assert "level 0 has a zero diagonal at row 37" in msg and msg == error_of(Zm, monkeypatch, host=True)
    D = sp.diags(np.arange(1.0, 301.0), format="csc")
    Dm = amg.CscMatrix(300, 300, D.indptr, D.indices, D.data)
    msg = error_of(Dm, monkeypatch, host=False)
    assert "level 0 does not reduce" in msg and msg == error_of(Dm, monkeypatch, host=True)


def test_coarse_stop_rule_matches_host_setup(monkeypatch):
    A = amg.Grid.laplacian(129)
    dev = build(A, "jacobi", monkeypatch, host=False, theta=0.15)
    ref = build(A, "jacobi", monkeypatch, host=True, theta=0.15)
    assert dev.n_levels == ref.n_levels == 6 and dev.get_n_dofs(5) == ref.get_n_dofs(5) > 200
    for l in range(6):
        assert same_csc(dev.get_coefficient_matrix(l), ref.get_coefficient_matrix(l)), l


def test_setup_times(monkeypatch):
    A = amg.Grid.laplacian(129)
    for host_setup in (False, True):
        t = build(A, "jacobi", monkeypatch, host_setup).setup_times()
        assert sorted(t) == sorted(("aggregation", "prolongators", "galerkin", "mirrors"))
        assert all(v > 0.0 for v in t.values()), t
    mg = amg.Multigrid(amg.LinearInterpolator(5), amg.DampedJacobi(), A, amg.Grid.rhs(129), 5)
    with pytest.raises(amg.AmgbError) as e:
        mg.setup_times()
    assert e.value.code == amg.ESTATE
