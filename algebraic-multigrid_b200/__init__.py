"""Thin ctypes binding of libamgb.so (include/amgb.h) for tests and bench.py.

The product is the CUDA library and its C ABI; the host-side mirror of the
reference's C++ interface lives in include/amg/*.hpp.  This module only gives
Python the same vocabulary (Grid, LinearInterpolator, SparseGaussSeidel,
Multigrid, rss -- /root/reference/include/amg/*.hpp) so that the parity tests
read like the reference's own test (test/testlib.cpp).  Nothing here computes:
every operation is a call into libamgb.so, and loading fails loudly when the
library has not been built.  The package directory name contains a hyphen;
import it with importlib.import_module("algebraic-multigrid_b200").
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libamgb.so")

OK, EINVAL, ECUDA, ENCCL, ESTATE = 0, 1, 2, 3, 4
SMOOTHER_GS, SMOOTHER_JACOBI, SMOOTHER_COLOR_GS, SMOOTHER_LINE_GS = 0, 1, 2, 3
LINES_X, LINES_Y, LINES_ALTERNATING = 0, 1, 2
GS_AUTO, GS_LEVELSCHED, GS_LINESCAN = 0, 1, 2
GS_KERNEL_FRONTS, GS_KERNEL_LINESCAN, GS_KERNEL_WAVE = 0, 1, 2
ARITH_REFERENCE, ARITH_FAST = 0, 1
TRANSFER_LINEAR, TRANSFER_BILINEAR_2D, TRANSFER_SMOOTHED_AGGREGATION = 0, 1, 2

_i, _l, _d, _p = C.c_int, C.c_int64, C.c_double, C.c_void_p
_pd = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")
_pi = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")


class Options(C.Structure):
    """amgb_options up to `lines`."""
    _fields_ = [("n_levels", _i), ("tolerance", _d),
                ("compute_error_every_n_iters", _l), ("n_iters", _l),
                ("smoother", _i), ("smoother_iters", _l), ("omega", _d),
                ("gs_mode", _i), ("use_graph", _i),
                ("skip_dead_coarse_smooth", _i), ("fuse", _i), ("arith", _i),
                ("transfer", _i), ("lines", _i)]


class FullOptions(C.Structure):
    """The whole amgb_options: Options, then the fields appended after `lines`.  sizeof(Options) is a
    multiple of 8, which is where the C struct's next double starts, so the layouts agree; the fields of
    Options are reachable directly (o.n_levels)."""
    _anonymous_ = ("base",)
    _fields_ = [("base", Options), ("strength", _d)]


class AmgbError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("amgb error %d: %s" % (code, msg))
        self.code = code


class InvalidArgument(AmgbError, ValueError):
    """AMGB_EINVAL -- the reference throws std::invalid_argument here."""


# every exported symbol of include/amgb.h: name -> (restype, argtypes)
SIGNATURES = {
    "amgb_last_error": (C.c_char_p, []),
    "amgb_version": (_i, []),
    "amgb_device_count": (_i, []),
    "amgb_set_device": (_i, [_i]),
    "amgb_grid_spacing_h": (_d, [_l]),
    "amgb_points_n_from_grid_spacing_h": (_l, [_d]),
    "amgb_grid_laplacian_nnz": (_l, [_l]),
    "amgb_grid_laplacian": (_i, [_l, _d, _pi, _pi, _pd]),
    "amgb_grid_rhs": (_i, [_l, _pd]),
    "amgb_n_H_dofs_from_n_h_dofs": (_l, [_l]),
    "amgb_interp_nnz": (_l, [_l, _l]),
    "amgb_interp_make_operators": (_i, [_l, _l, _pi, _pi, _pd, _pi, _pi, _pd]),
    "amgb_bilinear_coarse_lines": (_l, [_l]),
    "amgb_bilinear_nnz": (_l, [_l, _l]),
    "amgb_bilinear_make_operators": (_i, [_l, _l, _pi, _pi, _pd, _pi, _pi, _pd]),
    "amgb_sa_aggregate": (_i, [_i, _pi, _pi, _pd, _d, _pi, C.POINTER(_l)]),
    "amgb_linear_restrict": (_i, [_l, _l, _pd, _pd]),
    "amgb_linear_prolong": (_i, [_l, _l, _pd, _pd]),
    "amgb_csc_spmv": (_i, [_i, _i, _pi, _pi, _pd, _pd, _pd]),
    "amgb_csc_multiply": (_i, [_i, _i, _pi, _pi, _pd, _i, _pi, _pi, _pd, C.POINTER(_l), _p, _p, _p]),
    "amgb_matrix_create": (_i, [_i, _i, _pi, _pi, _pd, C.POINTER(_p)]),
    "amgb_matrix_destroy": (_i, [_p]),
    "amgb_matrix_nnz_device": (_l, [_p]),
    "amgb_matrix_is_symmetric": (_i, [_p]),
    "amgb_smooth_gs": (_i, [_p, _pd, _pd, _d, _l, _l, _i, C.POINTER(_l), C.POINTER(_d)]),
    "amgb_smooth_jacobi": (_i, [_p, _pd, _pd, _d, _l]),
    "amgb_smooth_color_gs": (_i, [_p, _pd, _pd, _l]),
    "amgb_smooth_line_gs": (_i, [_p, _pd, _pd, _l, _i]),
    "amgb_matrix_coloring": (_i, [_p, C.POINTER(_i), _pi]),
    "amgb_residual": (_i, [_p, _pd, _pd, _pd]),
    "amgb_rss": (_i, [_p, _pd, _pd, C.POINTER(_d)]),
    "amgb_matrix_time": (_i, [_p, _i, _d, _i, _i, C.POINTER(_d)]),
    "amgb_matrix_stream_bytes": (_l, [_p, _i]),
    "amgb_matrix_gs_kernel": (_i, [_p, _i]),
    "amgb_selftest_division": (_i, [_l, C.c_uint64, C.POINTER(_l)]),
    "amgb_options_default": (None, [C.POINTER(FullOptions)]),
    "amgb_hierarchy_create": (_i, [_i, _i, _pi, _pi, _pd, _pd, _l, C.POINTER(FullOptions),
                                   C.POINTER(_p)]),
    "amgb_hierarchy_destroy": (_i, [_p]),
    "amgb_hierarchy_transfer": (_i, [_p]),
    "amgb_hierarchy_get_transfer": (_i, [_p, _i, C.POINTER(_l), _p, _p, _p]),
    "amgb_hierarchy_device_setup": (_i, [_p]),
    "amgb_hierarchy_setup_times": (_i, [_p, _pd]),
    "amgb_comm_unique_id_bytes": (_i, []),
    "amgb_comm_get_unique_id": (_i, [_p]),
    "amgb_comm_create": (_i, [_p, _i, _i, C.POINTER(_p)]),
    "amgb_comm_destroy": (_i, [_p]),
    "amgb_hierarchy_create_sharded": (_i, [_p, _l, _i, _i, _pi, _pi, _pd, _pd, _l, C.POINTER(FullOptions),
                                           C.POINTER(_p)]),
    "amgb_hierarchy_n_sharded_levels": (_i, [_p]),
    "amgb_hierarchy_local_range": (_i, [_p, _i, C.POINTER(_l), C.POINTER(_l)]),
    "amgb_hierarchy_halo_exchanges_per_vcycle": (_l, [_p]),
    "amgb_hierarchy_halo_mode": (_i, [_p]),
    "amgb_hierarchy_halo_timed_out": (_i, [_p]),
    "amgb_partition_plan": (_i, [_i, np.ctypeslib.ndpointer(dtype=np.int64, flags="C_CONTIGUOUS"), _pi, _i, _l,
                                 C.POINTER(_i), np.ctypeslib.ndpointer(dtype=np.int64, flags="C_CONTIGUOUS"),
                                 _pi, _pi, _pi]),
    "amgb_partition_plan_2d": (_i, [_i, np.ctypeslib.ndpointer(dtype=np.int64, flags="C_CONTIGUOUS"), _i, _l,
                                    C.POINTER(_i), np.ctypeslib.ndpointer(dtype=np.int64, flags="C_CONTIGUOUS"),
                                    _pi, _pi, _pi]),
    "amgb_hierarchy_set_stream": (_i, [_p, _p]),
    "amgb_hierarchy_n_levels": (_i, [_p]),
    "amgb_hierarchy_n_dofs": (_l, [_p, _i]),
    "amgb_hierarchy_nnz": (_l, [_p, _i]),
    "amgb_hierarchy_nnz_device": (_l, [_p, _i]),
    "amgb_hierarchy_tolerance": (_d, [_p]),
    "amgb_hierarchy_get_matrix": (_i, [_p, _i, _pi, _pi, _pd]),
    "amgb_hierarchy_get_soln": (_i, [_p, _i, _p]),
    "amgb_hierarchy_get_rhs": (_i, [_p, _i, _p]),
    "amgb_hierarchy_set_soln": (_i, [_p, _i, _p]),
    "amgb_hierarchy_set_rhs": (_i, [_p, _i, _p]),
    "amgb_hierarchy_get_soln_local": (_i, [_p, _i, _p]),
    "amgb_hierarchy_get_rhs_local": (_i, [_p, _i, _p]),
    "amgb_hierarchy_set_soln_local": (_i, [_p, _i, _p]),
    "amgb_hierarchy_set_rhs_local": (_i, [_p, _i, _p]),
    "amgb_hierarchy_get_coloring": (_i, [_p, _i, C.POINTER(_i), _pi]),
    "amgb_vcycle": (_i, [_p]),
    "amgb_vcycles": (_i, [_p, _l]),
    "amgb_hierarchy_rss": (_i, [_p, C.POINTER(_d)]),
    "amgb_solve": (_i, [_p, C.POINTER(_l), C.POINTER(_d)]),
    "amgb_solve_relative": (_i, [_p, _d, C.POINTER(_l), C.POINTER(_d)]),
    "amgb_solve_pcg": (_i, [_p, _d, _l, C.POINTER(_l), C.POINTER(_d)]),
    "amgb_solve_gmres": (_i, [_p, _d, _i, _l, C.POINTER(_l), C.POINTER(_d)]),
    "amgb_hierarchy_iters_done": (_l, [_p]),
    "amgb_hierarchy_error_history": (_l, [_p, _pd, _l]),
    "amgb_synchronize": (_i, [_p]),
    "amgb_restrict": (_i, [_p, _i, _pd, _pd]),
    "amgb_prolong_add": (_i, [_p, _i, _pd, _pd]),
    "amgb_smooth_level": (_i, [_p, _i]),
    "amgb_residual_level": (_i, [_p, _i, _pd]),
    "amgb_residual_restrict_level": (_i, [_p, _i]),
    "amgb_coarse_solve": (_i, [_p]),
    "amgb_hierarchy_phase_times": (_i, [_p, _i, _pd]),
    "amgb_kernel_launches": (_l, []),
    "amgb_hierarchy_launches_per_vcycle": (_l, [_p]),
    "amgb_hierarchy_fused_legs": (_i, [_p, _i]),
    "amgb_hierarchy_matrix_free": (_i, [_p, _i]),
    "amgb_hierarchy_dictionary_types": (_i, [_p, _i]),
    "amgb_hierarchy_tail_first": (_i, [_p]),
    "amgb_hierarchy_mid_range": (_i, [_p, C.POINTER(_i), C.POINTER(_i), C.POINTER(_i), C.POINTER(_i)]),
    "amgb_hierarchy_galerkin_device": (_i, [_p, _i, C.POINTER(_d), C.POINTER(_l)]),
    "amgb_hierarchy_leg_plan": (_i, [_p, _i, _i, np.ctypeslib.ndpointer(dtype=np.int64, flags="C_CONTIGUOUS")]),
    "amgb_hierarchy_pass_bytes": (_l, [_p, _i]),
    "amgb_hierarchy_vcycle_bytes": (_l, [_p]),
    "amgb_hierarchy_format": (_i, [_p, _i]),
    "amgb_hierarchy_matrix_bytes": (_l, [_p, _i]),
    "amgb_hierarchy_n_diagonals": (_i, [_p, _i]),
    "amgb_hierarchy_gs_kernel": (_i, [_p, _i]),
    "amgb_time_kernel": (_i, [_p, _i, _i, _i, _i, C.POINTER(_d)]),
}

_lib = None


def lib():
    """Load libamgb.so; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                "libamgb.so is missing: build it with `python -c 'import __graft_entry__ as g; "
                "g.build()'` or `make -C algebraic-multigrid_b200/csrc`; there is no CPU fallback")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def _check(code):
    if code != OK:
        msg = lib().amgb_last_error().decode()
        raise (InvalidArgument if code == EINVAL else AmgbError)(code, msg)


def _f64(x):
    return np.ascontiguousarray(x, np.float64)


def _i32(x):
    return np.ascontiguousarray(x, np.int32)


def device_count():
    return lib().amgb_device_count()


def kernel_launches():
    return lib().amgb_kernel_launches()


class CscMatrix:
    """Host CSC triple with int32 indices (what Eigen::SparseMatrix<double> holds)."""

    def __init__(self, rows, cols, colptr, rowidx, val):
        self.rows, self.cols = int(rows), int(cols)
        self.colptr, self.rowidx, self.val = _i32(colptr), _i32(rowidx), _f64(val)

    @property
    def nnz(self):
        return int(self.colptr[-1])

    def to_scipy(self):
        import scipy.sparse as sp
        return sp.csc_matrix((self.val, self.rowidx, self.colptr), shape=(self.rows, self.cols))


class Grid:
    """AMG::Grid<double> (include/amg/grid.hpp:19-141)."""

    @staticmethod
    def grid_spacing_h(n):
        return lib().amgb_grid_spacing_h(n)

    @staticmethod
    def points_n_from_grid_spacing_h(h=1.0 / 50):
        return lib().amgb_points_n_from_grid_spacing_h(h)

    @staticmethod
    def laplacian(n, eps_y=1.0):
        nnz = lib().amgb_grid_laplacian_nnz(n)
        colptr = np.empty(n * n + 1, np.int32)
        rowidx = np.empty(nnz, np.int32)
        val = np.empty(nnz, np.float64)
        _check(lib().amgb_grid_laplacian(n, float(eps_y), colptr, rowidx, val))
        return CscMatrix(n * n, n * n, colptr, rowidx, val)

    @staticmethod
    def rhs(n):
        b = np.empty(n * n, np.float64)
        _check(lib().amgb_grid_rhs(n, b))
        return b


class LinearInterpolator:
    """AMG::LinearInterpolator<double> (include/amg/interpolator.hpp:98-141)."""

    def __init__(self, n_levels):
        self.n_levels = n_levels
        self._P = [None] * max(n_levels - 1, 0)
        self._R = [None] * max(n_levels - 1, 0)

    def make_operators(self, n_h, n_H, level):
        nnz = lib().amgb_interp_nnz(n_h, n_H)
        Pc, Pr, Pv = np.empty(n_H + 1, np.int32), np.empty(nnz, np.int32), np.empty(nnz)
        Rc, Rr, Rv = np.empty(n_h + 1, np.int32), np.empty(nnz, np.int32), np.empty(nnz)
        _check(lib().amgb_interp_make_operators(n_h, n_H, Pc, Pr, Pv, Rc, Rr, Rv))
        self._P[level] = CscMatrix(n_h, n_H, Pc, Pr, Pv)
        self._R[level] = CscMatrix(n_H, n_h, Rc, Rr, Rv)

    def get_P(self, level):
        return self._P[level]

    def get_R(self, level):
        return self._R[level]

    def set_level_to_P(self, level, P):
        self._P[level] = P

    def set_level_to_R(self, level, R):
        self._R[level] = R

    # interpolator.hpp:52-68: the STORED operators times the vector (generic device SpMV in
    # Eigen's order), whatever make_operators put there
    def prolongation(self, v, level):
        P = self._P[level]
        out = np.empty(P.rows)
        _check(lib().amgb_csc_spmv(P.rows, P.cols, P.colptr, P.rowidx, P.val, _f64(v), out))
        return out

    def restriction(self, v, level):
        R = self._R[level]
        out = np.empty(R.rows)
        _check(lib().amgb_csc_spmv(R.rows, R.cols, R.colptr, R.rowidx, R.val, _f64(v), out))
        return out


class BilinearInterpolator2D(LinearInterpolator):
    """Bilinear interpolation on an m x m grid of DOFs numbered k = y*m + x (TRANSFER_BILINEAR_2D):
    P = P1 (x) P1 with LinearInterpolator's 1-D pattern P1, m_H = m_h // 2 lines, R = P^T.  No
    reference counterpart: the 2-D coarsening that makes the V-cycle converge independently of the
    grid size on 2-D problems, where the reference's 1-D rule semi-coarsens the flattened vector."""

    transfer = TRANSFER_BILINEAR_2D

    @staticmethod
    def coarse_lines(m_h):
        return lib().amgb_bilinear_coarse_lines(m_h)

    def make_operators(self, n_h, n_H, level):
        m_h, m_H = int(round(n_h ** 0.5)), int(round(n_H ** 0.5))
        if m_h * m_h != n_h or m_H * m_H != n_H or m_H != self.coarse_lines(m_h):
            raise InvalidArgument(EINVAL, "BilinearInterpolator2D: %d -> %d DOFs are not m^2 -> (m // 2)^2"
                                  % (n_h, n_H))
        nnz = lib().amgb_bilinear_nnz(m_h, m_H)
        Pc, Pr, Pv = np.empty(n_H + 1, np.int32), np.empty(nnz, np.int32), np.empty(nnz)
        Rc, Rr, Rv = np.empty(n_h + 1, np.int32), np.empty(nnz, np.int32), np.empty(nnz)
        _check(lib().amgb_bilinear_make_operators(m_h, m_H, Pc, Pr, Pv, Rc, Rr, Rv))
        self._P[level] = CscMatrix(n_h, n_H, Pc, Pr, Pv)
        self._R[level] = CscMatrix(n_H, n_h, Rc, Rr, Rv)


class SmoothedAggregation(LinearInterpolator):
    """Smoothed-aggregation coarsening (TRANSFER_SMOOTHED_AGGREGATION, include/amgb.h): aggregates of
    strongly coupled rows (threshold `strength`), P = (I - w D^-1 A) T.  Needs no grid, so it runs on
    rectangular grids, permuted numberings, wide stencils and unstructured matrices.  n_levels is a cap:
    the hierarchy coarsens while a level has more than 200 rows, and stops at a coarse level whose
    aggregation does not reduce it.  The aggregation depends on A, so
    Multigrid fills the P and R slots from the hierarchy it built; make_operators cannot."""

    transfer = TRANSFER_SMOOTHED_AGGREGATION

    def __init__(self, n_levels, strength=0.08):
        super().__init__(n_levels)
        self.strength = float(strength)

    def make_operators(self, n_h, n_H, level):
        raise NotImplementedError("SmoothedAggregation's operators depend on A: Multigrid builds them")


def sa_aggregate(A, strength=0.08):
    """(agg, n_aggregates) of the smoothed-aggregation rule on host matrix A (host only)."""
    agg = np.empty(A.cols, np.int32)
    k = _l()
    _check(lib().amgb_sa_aggregate(A.cols, A.colptr, A.rowidx, A.val, float(strength), agg, C.byref(k)))
    return agg, k.value


def csc_multiply(A, B):
    """A @ B of two CscMatrix on the device, in the order of the smoothed-aggregation setup's products: each
    entry sums over ascending inner index, the first term initialising the sum; structural and computed
    zeros are kept and every column comes out sorted."""
    if A.cols != B.rows:
        raise InvalidArgument(EINVAL, "csc_multiply: inner dimensions differ (%d x %d times %d x %d)"
                              % (A.rows, A.cols, B.rows, B.cols))
    nnz = _l()
    args = (A.rows, A.cols, A.colptr, A.rowidx, A.val, B.cols, B.colptr, B.rowidx, B.val, C.byref(nnz))
    _check(lib().amgb_csc_multiply(*args, None, None, None))
    colptr, rowidx, val = np.empty(B.cols + 1, np.int32), np.empty(nnz.value, np.int32), np.empty(nnz.value)
    _check(lib().amgb_csc_multiply(*args, colptr.ctypes.data, rowidx.ctypes.data, val.ctypes.data))
    return CscMatrix(A.rows, B.cols, colptr, rowidx, val)


def _transpose(M):
    """CSC of M^T (an index permutation: entries keep their values, rows stay ascending).  scipy's CSC -> CSR
    conversion is a stable counting sort, linear in the entries."""
    import scipy.sparse as sp
    T = sp.csc_matrix((M.val, M.rowidx, M.colptr), shape=(M.rows, M.cols)).tocsr()
    return CscMatrix(M.cols, M.rows, T.indptr, T.indices, T.data)


class DeviceMatrix:
    """Device mirror of one CSC matrix (amgb_matrix)."""

    def __init__(self, A):
        self.A = A
        h = _p()
        _check(lib().amgb_matrix_create(A.rows, A.cols, A.colptr, A.rowidx, A.val, C.byref(h)))
        self.h = h

    def __del__(self):
        if getattr(self, "h", None) and _lib is not None:
            _lib.amgb_matrix_destroy(self.h)
            self.h = None

    @property
    def nnz_device(self):
        return lib().amgb_matrix_nnz_device(self.h)

    @property
    def is_symmetric(self):
        return bool(lib().amgb_matrix_is_symmetric(self.h))

    def residual(self, u, f):
        r = np.empty(self.A.rows)
        _check(lib().amgb_residual(self.h, _f64(u), _f64(f), r))
        return r

    def rss(self, u, b):
        out = _d()
        _check(lib().amgb_rss(self.h, _f64(u), _f64(b), C.byref(out)))
        return out.value

    def coloring(self):
        nc = _i()
        color = np.empty(self.A.cols, np.int32)
        _check(lib().amgb_matrix_coloring(self.h, C.byref(nc), color))
        return nc.value, color

    def time_pass(self, kind, omega=2.0 / 3.0, warmup=3, reps=10):
        """ms per launch of one Jacobi sweep (0) / colour-complete sweep (1) / residual (2) on the
        vectors the last residual() / rss() call uploaded."""
        ms = _d()
        _check(lib().amgb_matrix_time(self.h, kind, omega, warmup, reps, C.byref(ms)))
        return ms.value

    def stream_bytes(self, kind):
        return lib().amgb_matrix_stream_bytes(self.h, kind)

    def gs_kernel(self, mode=GS_AUTO):
        """GS_KERNEL_* the lexicographic Gauss-Seidel mode runs on this matrix."""
        k = lib().amgb_matrix_gs_kernel(self.h, mode)
        if k < 0:
            raise AmgbError(lib().amgb_last_error().decode())
        return k


def _fingerprint(A):
    """Content fingerprint of a host CSC matrix: every byte of colptr / rowidx / val when the
    matrix has at most 4 M entries, else 65536 evenly spaced entries of each array (a changed
    value between the samples is not seen: call invalidate_mirror(A) after editing a large
    matrix in place)."""
    import zlib
    nnz = A.nnz
    if nnz <= (1 << 22):
        parts = (A.colptr, A.rowidx, A.val)
    else:
        step = max(1, nnz // 65536)
        parts = (A.colptr[::max(1, A.colptr.shape[0] // 65536)], A.rowidx[::step], A.val[::step])
    h = 0
    for a in parts:
        h = zlib.crc32(np.ascontiguousarray(a).view(np.uint8), h)
    return (A.rows, A.cols, nnz, h)


def invalidate_mirror(A):
    """Drop the cached device mirror of A (after its values were changed in place)."""
    A._amgb_mirror = None


def _mirror(A):
    """Device mirror of a host matrix, cached on the object and re-validated against a content
    fingerprint on every use: values edited in place give a fresh upload, not a stale mirror
    (the reference always reads the live matrix)."""
    if isinstance(A, DeviceMatrix):
        return A
    fp = _fingerprint(A)
    cached = getattr(A, "_amgb_mirror", None)
    if cached is None or cached[0] != fp:
        cached = (fp, DeviceMatrix(A))
        A._amgb_mirror = cached
    return cached[1]


def selftest_division(n_pairs=1 << 24, seed=1):
    """Mismatches between the wavefront kernel's split division and the compiler's IEEE division."""
    bad = _l()
    _check(lib().amgb_selftest_division(n_pairs, seed, C.byref(bad)))
    return bad.value


def rss(A, u, b):
    """AMG::rss (include/amg/common.hpp:17-27)."""
    return _mirror(A).rss(u, b)


class SmootherBase:
    """AMG::SmootherBase<double> (include/amg/smoother.hpp:18-66)."""
    kind = None

    def __init__(self, *args):
        self.tolerance = 1e-9
        self.compute_error_every_n_iters = 100
        self.n_iters = 1
        if len(args) == 1:
            self.n_iters = int(args[0])
        elif len(args) == 3:
            self.tolerance, self.compute_error_every_n_iters, self.n_iters = (
                float(args[0]), int(args[1]), int(args[2]))
        elif len(args) != 0:
            raise TypeError("SmootherBase(), SmootherBase(n_iters) or "
                            "SmootherBase(tolerance, compute_error_every_n_iters, n_iters)")
        self.iters_done = 0
        self.last_error = 100.0


class SparseGaussSeidel(SmootherBase):
    """AMG::SparseGaussSeidel<double> (include/amg/smoother.hpp:86-216)."""
    kind = SMOOTHER_GS

    def __init__(self, *args, mode=GS_AUTO):
        super().__init__(*args)
        if len(args) == 0:  # smoother.hpp:183-187
            self.tolerance, self.compute_error_every_n_iters, self.n_iters = 1e-9, 0, 1
        self.mode = mode

    def smooth(self, A, u, b):
        """u is updated in place."""
        it, err = _l(), _d()
        _check(lib().amgb_smooth_gs(_mirror(A).h, u, _f64(b), self.tolerance,
                                    self.compute_error_every_n_iters, self.n_iters, self.mode,
                                    C.byref(it), C.byref(err)))
        self.iters_done, self.last_error = it.value, err.value
        if self.compute_error_every_n_iters != 0:  # smoother.hpp:205-212
            print("SPGS %s after %d iterations." % (
                "converged" if err.value <= self.tolerance else "did not converge", it.value))


class DampedJacobi(SmootherBase):
    """u <- u + omega D^-1 (f - A u), n_iters sweeps per smooth() (no reference counterpart)."""
    kind = SMOOTHER_JACOBI

    def __init__(self, omega=2.0 / 3.0, n_iters=2):
        super().__init__(n_iters)
        self.omega = omega

    def smooth(self, A, u, b):
        _check(lib().amgb_smooth_jacobi(_mirror(A).h, u, _f64(b), self.omega, self.n_iters))


class MulticolorGaussSeidel(SmootherBase):
    """Greedy multicolour symmetric Gauss-Seidel (red-black on the 5-point level)."""
    kind = SMOOTHER_COLOR_GS

    def __init__(self, n_iters=1):
        super().__init__(n_iters)

    def smooth(self, A, u, b):
        _check(lib().amgb_smooth_color_gs(_mirror(A).h, u, _f64(b), self.n_iters))


class LineGaussSeidel(SmootherBase):
    """Zebra line Gauss-Seidel on an m x m grid operator (include/amgb.h, AMGB_SMOOTHER_LINE_GS);
    `lines` is LINES_X (strong x-coupling), LINES_Y or LINES_ALTERNATING.  Multigrid needs a
    BilinearInterpolator2D with it."""
    kind = SMOOTHER_LINE_GS

    def __init__(self, n_iters=1, lines=LINES_X):
        super().__init__(n_iters)
        if lines not in (LINES_X, LINES_Y, LINES_ALTERNATING):
            raise ValueError("`lines` must be LINES_X, LINES_Y or LINES_ALTERNATING, got %r" % (lines,))
        self.lines = lines

    def smooth(self, A, u, b):
        _check(lib().amgb_smooth_line_gs(_mirror(A).h, u, _f64(b), self.n_iters, self.lines))


class Comm:
    """One NCCL communicator per process (amgb_comm).  `exchange_id` is a callable that
    takes rank 0's id bytes (or None on other ranks) and returns rank 0's bytes on every
    rank -- e.g. a torch.distributed broadcast; the library itself never imports torch."""

    def __init__(self, rank, world, exchange_id):
        nbytes = lib().amgb_comm_unique_id_bytes()
        buf = C.create_string_buffer(nbytes)
        if rank == 0:
            _check(lib().amgb_comm_get_unique_id(buf))
        raw = exchange_id(buf.raw if rank == 0 else None)
        buf = C.create_string_buffer(bytes(raw), nbytes)
        h = _p()
        _check(lib().amgb_comm_create(buf, rank, world, C.byref(h)))
        self.h, self.rank, self.world = h, rank, world

    def __del__(self):
        if getattr(self, "h", None) and _lib is not None:
            _lib.amgb_comm_destroy(self.h)
            self.h = None


def partition_plan(level_sizes, half_bandwidth, world, min_rows_per_rank):
    """Host-only: (n_sharded, starts[l][g], halo_lo, halo_hi, ghost) of the row-block plan."""
    L = len(level_sizes)
    sizes = np.ascontiguousarray(level_sizes, np.int64)
    bw = _i32(half_bandwidth)
    ns = _i()
    starts = np.zeros(L * (world + 1), np.int64)
    lo, hi, gh = np.zeros(L, np.int32), np.zeros(L, np.int32), np.zeros(L, np.int32)
    _check(lib().amgb_partition_plan(L, sizes, bw, world, min_rows_per_rank, C.byref(ns), starts, lo, hi, gh))
    k = ns.value
    return k, starts.reshape(L, world + 1)[:k], lo[:k], hi[:k], gh[:k]


def partition_plan_2d(lines, world, min_rows_per_rank):
    """Host-only: (n_sharded, starts[l][g], halo_lo, halo_hi, ghost), all in rows, of the plan of a
    bilinear 2-D hierarchy with `lines[l]` grid lines on level l (blocks of whole lines)."""
    L = len(lines)
    m = np.ascontiguousarray(lines, np.int64)
    ns = _i()
    starts = np.zeros(L * (world + 1), np.int64)
    lo, hi, gh = np.zeros(L, np.int32), np.zeros(L, np.int32), np.zeros(L, np.int32)
    _check(lib().amgb_partition_plan_2d(L, m, world, min_rows_per_rank, C.byref(ns), starts, lo, hi, gh))
    k = ns.value
    return k, starts.reshape(L, world + 1)[:k], lo[:k], hi[:k], gh[:k]


class Multigrid:
    """AMG::Multigrid<double> (include/amg/multigrid.hpp:22-365) on the device."""

    def __init__(self, interpolator, smoother, A, b, n_levels, tolerance=1e-9,
                 compute_error_every_n_iters=10, n_iters=100, use_graph=True,
                 skip_dead_coarse_smooth=True, comm=None, min_rows_per_rank=1 << 18, fuse=None,
                 arith=ARITH_REFERENCE):
        self.interpolator, self.smoother = interpolator, smoother
        o = FullOptions()
        lib().amgb_options_default(C.byref(o))
        o.n_levels = n_levels
        o.tolerance = tolerance
        o.compute_error_every_n_iters = compute_error_every_n_iters
        o.n_iters = n_iters
        o.smoother = smoother.kind
        o.smoother_iters = smoother.n_iters
        o.omega = getattr(smoother, "omega", 2.0 / 3.0)
        o.gs_mode = getattr(smoother, "mode", GS_AUTO)
        o.use_graph = int(use_graph)
        o.skip_dead_coarse_smooth = int(skip_dead_coarse_smooth)
        if fuse is not None:
            o.fuse = int(fuse)
        o.arith = int(arith)
        o.transfer = int(getattr(interpolator, "transfer", TRANSFER_LINEAR))
        o.lines = int(getattr(smoother, "lines", LINES_X))
        o.strength = float(getattr(interpolator, "strength", o.strength))
        b = _f64(b)
        h = _p()
        if comm is None:
            _check(lib().amgb_hierarchy_create(A.rows, A.cols, A.colptr, A.rowidx, A.val, b, b.shape[0],
                                               C.byref(o), C.byref(h)))
        else:
            _check(lib().amgb_hierarchy_create_sharded(comm.h, min_rows_per_rank, A.rows, A.cols, A.colptr,
                                                       A.rowidx, A.val, b, b.shape[0], C.byref(o),
                                                       C.byref(h)))
        self.comm = comm
        self.h = h
        self.n_levels = lib().amgb_hierarchy_n_levels(h)  # (a cap for smoothed aggregation)
        self.display_error = False
        # the driver fills the interpolator's slots like the reference does (multigrid.hpp:218)
        if interpolator is not None:
            for l in range(1, self.n_levels):
                if o.transfer == TRANSFER_SMOOTHED_AGGREGATION:
                    P = self.get_transfer(l - 1)
                    interpolator.set_level_to_P(l - 1, P)
                    interpolator.set_level_to_R(l - 1, _transpose(P))
                else:
                    interpolator.make_operators(self.get_n_dofs(l - 1), self.get_n_dofs(l), l - 1)

    def __del__(self):
        if getattr(self, "h", None) and _lib is not None:
            _lib.amgb_hierarchy_destroy(self.h)
            self.h = None

    # ---- reference getters (multigrid.hpp:339-354) ----
    def get_n_dofs(self, level):
        return lib().amgb_hierarchy_n_dofs(self.h, level)

    def transfer(self):
        """TRANSFER_* the hierarchy was built with."""
        return lib().amgb_hierarchy_transfer(self.h)

    def get_transfer(self, level):
        """P of `level` (n_level x n_level+1) as the hierarchy applies it."""
        nnz = _l()
        _check(lib().amgb_hierarchy_get_transfer(self.h, level, C.byref(nnz), None, None, None))
        nf, nc = self.get_n_dofs(level), self.get_n_dofs(level + 1)
        colptr, rowidx, val = np.empty(nc + 1, np.int32), np.empty(nnz.value, np.int32), np.empty(nnz.value)
        _check(lib().amgb_hierarchy_get_transfer(self.h, level, C.byref(nnz), colptr.ctypes.data,
                                                 rowidx.ctypes.data, val.ctypes.data))
        return CscMatrix(nf, nc, colptr, rowidx, val)

    @property
    def device_setup(self):
        """True when the level operators were built on the GPU (AMGB_HOST_SETUP=1 forces the host setup)."""
        return bool(lib().amgb_hierarchy_device_setup(self.h))

    def setup_times(self):
        """Seconds of the setup phases of a smoothed-aggregation hierarchy (host clock, each phase ending in a
        stream synchronise)."""
        out = np.zeros(4)
        _check(lib().amgb_hierarchy_setup_times(self.h, out))
        return dict(zip(("aggregation", "prolongators", "galerkin", "mirrors"), out.tolist()))

    def get_tolerance(self):
        return lib().amgb_hierarchy_tolerance(self.h)

    def get_coefficient_matrix(self, level):
        n = self.get_n_dofs(level)
        nnz = lib().amgb_hierarchy_nnz(self.h, level)
        colptr, rowidx, val = np.empty(n + 1, np.int32), np.empty(nnz, np.int32), np.empty(nnz)
        _check(lib().amgb_hierarchy_get_matrix(self.h, level, colptr, rowidx, val))
        return CscMatrix(n, n, colptr, rowidx, val)

    def get_soln(self, level, out=None):
        u = np.empty(self.get_n_dofs(level)) if out is None else out
        _check(lib().amgb_hierarchy_get_soln(self.h, level, u.ctypes.data))
        return u

    def get_rhs(self, level, out=None):
        f = np.empty(self.get_n_dofs(level)) if out is None else out
        _check(lib().amgb_hierarchy_get_rhs(self.h, level, f.ctypes.data))
        return f

    def set_soln(self, level, u):
        u = _f64(u)
        assert u.shape[0] == self.get_n_dofs(level)
        _check(lib().amgb_hierarchy_set_soln(self.h, level, u.ctypes.data))

    def set_rhs(self, level, f):
        f = _f64(f)
        assert f.shape[0] == self.get_n_dofs(level)
        _check(lib().amgb_hierarchy_set_rhs(self.h, level, f.ctypes.data))

    # ---- row-block variants (sharded hierarchies): this rank's rows of local_range only ----
    def get_soln_local(self, level, out=None):
        b, e = self.local_range(level)
        u = np.empty(e - b) if out is None else out
        _check(lib().amgb_hierarchy_get_soln_local(self.h, level, u.ctypes.data))
        return u

    def get_rhs_local(self, level, out=None):
        b, e = self.local_range(level)
        f = np.empty(e - b) if out is None else out
        _check(lib().amgb_hierarchy_get_rhs_local(self.h, level, f.ctypes.data))
        return f

    def set_soln_local(self, level, u):
        u = _f64(u)
        b, e = self.local_range(level)
        assert u.shape[0] == e - b
        _check(lib().amgb_hierarchy_set_soln_local(self.h, level, u.ctypes.data))

    def set_rhs_local(self, level, f):
        f = _f64(f)
        b, e = self.local_range(level)
        assert f.shape[0] == e - b
        _check(lib().amgb_hierarchy_set_rhs_local(self.h, level, f.ctypes.data))

    def display_error_on(self):
        self.display_error = True

    def display_error_off(self):
        # the reference sets the flag to true here (multigrid.hpp:361-364); this mirror
        # deliberately does what the name says
        self.display_error = False

    # ---- hot path ----
    def vcycle(self):
        _check(lib().amgb_vcycle(self.h))

    def vcycles(self, n):
        _check(lib().amgb_vcycles(self.h, n))

    def synchronize(self):
        _check(lib().amgb_synchronize(self.h))

    def rss(self):
        out = _d()
        _check(lib().amgb_hierarchy_rss(self.h, C.byref(out)))
        return out.value

    def solve(self):
        it, err = _l(), _d()
        _check(lib().amgb_solve(self.h, C.byref(it), C.byref(err)))
        self.iters_done, self.last_error = it.value, err.value
        if self.display_error:
            every = max(1, self.iters_done // max(1, len(self.error_history())))
            for k, e in enumerate(self.error_history()):
                print("Iter: %d | Error: %g" % ((k + 1) * every, e))
        print("AMG %s after %d iterations." % (
            "converged" if err.value <= self.get_tolerance() else "did not converge", it.value))
        return self.get_soln(0)

    def solve_relative(self, rel_tol):
        it, rel = _l(), _d()
        _check(lib().amgb_solve_relative(self.h, rel_tol, C.byref(it), C.byref(rel)))
        self.iters_done, self.last_error = it.value, rel.value
        return self.get_soln(0)

    def solve_pcg(self, rel_tol, max_iters=1000):
        """Conjugate gradients preconditioned by one V-cycle (beyond the reference)."""
        it, rel = _l(), _d()
        _check(lib().amgb_solve_pcg(self.h, rel_tol, max_iters, C.byref(it), C.byref(rel)))
        self.iters_done, self.last_error = it.value, rel.value
        return self.get_soln(0)

    def solve_gmres(self, rel_tol, restart=30, max_iters=1000):
        """Restarted GMRES(restart) right-preconditioned by one V-cycle, for symmetric and unsymmetric A alike
        (beyond the reference).  iters_done counts Arnoldi steps; last_error is the true relative residual."""
        it, rel = _l(), _d()
        _check(lib().amgb_solve_gmres(self.h, rel_tol, restart, max_iters, C.byref(it), C.byref(rel)))
        self.iters_done, self.last_error = it.value, rel.value
        return self.get_soln(0)

    def error_history(self):
        n = lib().amgb_hierarchy_error_history(self.h, np.empty(1), 0)
        out = np.empty(max(n, 1))
        lib().amgb_hierarchy_error_history(self.h, out, n)
        return out[:n]

    # ---- per-operator entry points ----
    def restrict(self, level, r_fine):
        out = np.empty(self.get_n_dofs(level + 1))
        _check(lib().amgb_restrict(self.h, level, _f64(r_fine), out))
        return out

    def prolong_add(self, level, e_coarse, u_fine):
        u = _f64(u_fine).copy()
        _check(lib().amgb_prolong_add(self.h, level, _f64(e_coarse), u))
        return u

    def smooth_level(self, level):
        _check(lib().amgb_smooth_level(self.h, level))

    def residual_level(self, level):
        r = np.empty(self.get_n_dofs(level))
        _check(lib().amgb_residual_level(self.h, level, r))
        return r

    def residual_restrict_level(self, level):
        _check(lib().amgb_residual_restrict_level(self.h, level))

    def coarse_solve(self):
        _check(lib().amgb_coarse_solve(self.h))

    def coloring(self, level):
        nc = _i()
        color = np.empty(self.get_n_dofs(level), np.int32)
        _check(lib().amgb_hierarchy_get_coloring(self.h, level, C.byref(nc), color))
        return nc.value, color

    # ---- sharding ----
    def n_sharded_levels(self):
        return lib().amgb_hierarchy_n_sharded_levels(self.h)

    def local_range(self, level):
        b, e = _l(), _l()
        _check(lib().amgb_hierarchy_local_range(self.h, level, C.byref(b), C.byref(e)))
        return b.value, e.value

    def halo_exchanges_per_vcycle(self):
        return lib().amgb_hierarchy_halo_exchanges_per_vcycle(self.h)

    def halo_mode(self):
        return {0: "none", 1: "nccl", 2: "peer"}[lib().amgb_hierarchy_halo_mode(self.h)]

    def halo_timed_out(self):
        return bool(lib().amgb_hierarchy_halo_timed_out(self.h))

    # ---- measurement helpers ----
    def set_stream(self, cuda_stream):
        _check(lib().amgb_hierarchy_set_stream(self.h, _p(cuda_stream)))

    def nnz(self, level):
        return lib().amgb_hierarchy_nnz(self.h, level)

    def nnz_device(self, level):
        return lib().amgb_hierarchy_nnz_device(self.h, level)

    def format(self, level):
        return {0: "sell", 1: "dia"}[lib().amgb_hierarchy_format(self.h, level)]

    def matrix_bytes(self, level):
        return lib().amgb_hierarchy_matrix_bytes(self.h, level)

    def n_diagonals(self, level):
        """Diagonals a fused leg streams per row: every diagonal of the DIA mirror, or the centre and
        upper ones on a level whose register-streaming legs read a bitwise-symmetric operator."""
        return lib().amgb_hierarchy_n_diagonals(self.h, level)

    def gs_kernel(self, level):
        """GS_KERNEL_* smoothing `level` (-1 unless the smoother is SparseGaussSeidel)."""
        return lib().amgb_hierarchy_gs_kernel(self.h, level)

    def pass_bytes(self, level):
        return lib().amgb_hierarchy_pass_bytes(self.h, level)

    def vcycle_bytes(self):
        return lib().amgb_hierarchy_vcycle_bytes(self.h)

    def launches_per_vcycle(self):
        return lib().amgb_hierarchy_launches_per_vcycle(self.h)

    def fused_legs(self, level):
        """True when `level` runs as one fused kernel per leg (option fuse bit 2)."""
        return bool(lib().amgb_hierarchy_fused_legs(self.h, level))

    def matrix_free(self, level):
        """True when the level's fused legs run matrix-free (verified constant five-point stencil)."""
        return bool(lib().amgb_hierarchy_matrix_free(self.h, level))

    def dictionary_types(self, level):
        """Distinct operator rows when the level's legs run from a row-type dictionary, else 0."""
        return lib().amgb_hierarchy_dictionary_types(self.h, level)

    def galerkin_device(self, level):
        """(kernel ms, entries differing from the host-built level + 1) of the device-side R (A P)."""
        ms, bad = _d(), _l()
        _check(lib().amgb_hierarchy_galerkin_device(self.h, level, C.byref(ms), C.byref(bad)))
        return ms.value, bad.value

    def phase_times(self, reps=10):
        """ms of [sharded down legs, gather, levels below the sharded ones, sharded up legs] on this rank."""
        out = np.zeros(4)
        _check(lib().amgb_hierarchy_phase_times(self.h, reps, out))
        return dict(zip(("sharded_down", "gather", "coarse_part", "sharded_up"), out.tolist()))

    def tail_first(self):
        """First level of the coarse tail that runs in one launch (-1: none)."""
        return lib().amgb_hierarchy_tail_first(self.h)

    def mid_range(self):
        """(first, end, tile rows, blocks) of the levels the two mid-level kernels cover; first = -1: none."""
        a, b, t, nb = _i(), _i(), _i(), _i()
        _check(lib().amgb_hierarchy_mid_range(self.h, C.byref(a), C.byref(b), C.byref(t), C.byref(nb)))
        return a.value, b.value, t.value, nb.value

    def leg_plan(self, level, up=False):
        info = np.zeros(10, np.int64)
        _check(lib().amgb_hierarchy_leg_plan(self.h, level, int(up), info))
        keys = ("m", "rho", "W", "LJ", "tiles", "strips", "PF", "threads", "smem_bytes", "NS")
        return dict(zip(keys, info.tolist()))

    def time_kernel(self, level, kind, warmup=3, reps=10):
        ms = _d()
        _check(lib().amgb_time_kernel(self.h, level, kind, warmup, reps, C.byref(ms)))
        return ms.value
