"""Worker for the multi-GPU test of the sharded bilinear 2-D hierarchy (launched with
torch.distributed.run, one rank per GPU).  Each rank builds the line-block sharded hierarchy, runs
V-cycles and compares every level's gathered iterate with the single-GPU 2-D hierarchy -- every kernel
is per-operator on both sides, so the bits must be identical in both arithmetic modes -- and with the
2-D oracle (tests/oracle_bilinear2d.py)."""
import importlib
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import oracle as O  # noqa: E402
import oracle_bilinear2d as O2  # noqa: E402

amg = importlib.import_module("algebraic-multigrid_b200")
REF, FAST = amg.ARITH_REFERENCE, amg.ARITH_FAST


def id_exchanger(raw):
    box = [raw]
    dist.broadcast_object_list(box, src=0)
    return box[0]


def smoother(nu):
    """nu > 0: damped Jacobi with nu sweeps; nu < 0: multicolour Gauss-Seidel with -nu symmetric sweeps."""
    return amg.MulticolorGaussSeidel(-nu) if nu < 0 else amg.DampedJacobi(2.0 / 3.0, nu)


def run_case(comm, rank, world, m, L, eps, min_rows, nu, fuse, arith, oracle):
    A, b = amg.Grid.laplacian(m, eps), amg.Grid.rhs(m)
    want_mode = os.environ.get("AMGB_HALO", "peer")
    for use_graph in (False, True):
        kw = dict(use_graph=use_graph, fuse=fuse, arith=arith)
        mg = amg.Multigrid(amg.BilinearInterpolator2D(L), smoother(nu), A, b, L, 1e-9, 1, 1, comm=comm,
                           min_rows_per_rank=min_rows, **kw)
        single = amg.Multigrid(amg.BilinearInterpolator2D(L), smoother(nu), A, b, L, 1e-9, 1, 1, **kw)
        ns = mg.n_sharded_levels()
        assert ns >= 1, ns
        assert mg.halo_mode() == want_mode, (mg.halo_mode(), want_mode)
        for _ in range(3):
            mg.vcycle()
            single.vcycle()
        for l in range(L):
            got, want = mg.get_soln(l), single.get_soln(l)
            assert got.tobytes() == want.tobytes(), (m, l, use_graph, nu, fuse, arith, np.abs(got - want).max())
        assert not mg.halo_timed_out()
        assert mg.halo_exchanges_per_vcycle() > 0
        r_sh, r_one = mg.rss(), single.rss()
        assert abs(r_sh - r_one) <= 1e-13 * r_one, (r_sh, r_one)
        # row-block getters / setters: this rank's rows only, and a cycle from the state they set
        b0, b1 = mg.local_range(0)
        assert b0 % m == 0 and b1 % m == 0
        assert mg.get_soln_local(0).tobytes() == single.get_soln(0)[b0:b1].tobytes()
        rng = np.random.default_rng(7)
        u_new, f_new = rng.standard_normal(m * m), rng.standard_normal(m * m)
        mg.set_soln_local(0, u_new[b0:b1]); mg.set_rhs_local(0, f_new[b0:b1])
        single.set_soln(0, u_new); single.set_rhs(0, f_new)
        mg.vcycle(); single.vcycle()
        assert mg.get_soln_local(0).tobytes() == single.get_soln(0)[b0:b1].tobytes()
        assert mg.get_rhs_local(0).tobytes() == f_new[b0:b1].tobytes()
        for l in range(L):
            assert mg.get_soln(l).tobytes() == single.get_soln(l).tobytes(), ("after set_*_local", l)
        mg.set_soln(0, np.zeros(m * m)); mg.set_rhs(0, b)
        if oracle and rank == 0 and not use_graph:
            mo = O2.Multigrid(O.laplacian(m, eps), b, L, 1e-9, 1, 1,
                              O.SMOOTHER_COLOR_GS if nu < 0 else O.SMOOTHER_JACOBI, abs(nu), 2.0 / 3.0)
            for _ in range(3):
                mo.vcycle()
                mg.vcycle()
            assert np.linalg.norm(mg.get_soln(0) - mo.u(0)) <= 1e-12 * np.linalg.norm(mo.u(0))
        else:
            for _ in range(3):
                mg.vcycle()
            mg.get_soln(0)  # collective: every rank takes part
        exchanges = mg.halo_exchanges_per_vcycle()
        del mg, single
        if use_graph:  # same cycle count to ||r|| / ||b|| <= 1e-8 (or the cap of 60) as one GPU
            its = []
            for c in (comm, None):
                h = amg.Multigrid(amg.BilinearInterpolator2D(L), smoother(nu), A, b, L, 1e-9, 1, 60, comm=c,
                                  min_rows_per_rank=min_rows, **kw)
                h.solve_relative(1e-8)
                its.append((h.iters_done, h.last_error))
                del h
            assert its[0][0] == its[1][0] and abs(its[0][1] - its[1][1]) <= 1e-12 * its[1][1], its
        if rank == 0:
            print("ok m=%d L=%d eps=%g sharded_levels=%d nu=%d fuse=%s arith=%d graph=%s halo=%s exchanges/vcycle=%d "
                  "rss=%.6e%s" % (m, L, eps, ns, nu, fuse, arith, use_graph, want_mode, exchanges, r_sh,
                                  " cycles_to_1e-8=%d" % its[0][0] if use_graph else ""), flush=True)


def check_rejections(comm):
    A, b = amg.Grid.laplacian(64), amg.Grid.rhs(64)
    for sm in (amg.LineGaussSeidel(1), amg.SparseGaussSeidel()):
        try:
            amg.Multigrid(amg.BilinearInterpolator2D(4), sm, A, b, 4, comm=comm, min_rows_per_rank=1)
        except ValueError:
            continue
        raise AssertionError("a sharded 2-D create with %s was accepted" % type(sm).__name__)


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    amg.lib().amgb_set_device(local)
    dist.init_process_group("gloo")
    comm = amg.Comm(rank, world, id_exchanger)
    # (m, levels, eps_y, min rows per rank, sweeps (< 0: multicolour GS), fuse option or None, arithmetic)
    cases = [(257, 6, 1.0, 4096, 2, None, REF),
             (256, 6, 1.0, 4096, 2, None, FAST),
             (513, 7, 1e-3, 8192, 2, 0, REF),      # zero-guess first sweep off
             (257, 6, 1e-3, 4096, 1, None, FAST),
             (256, 6, 1.0, 4096, 3, 0, REF),
             (257, 6, 1.0, 4096, -1, None, REF),   # multicolour GS: one exchange per colour pass
             (256, 6, 1e-3, 4096, -1, None, FAST),
             (513, 7, 1.0, 700, 2, None, REF),     # three or four sharded levels
             (300, 6, 1.0, 700, 2, None, FAST)]    # three sharded levels, uneven blocks
    if len(sys.argv) > 1 and sys.argv[1] == "big":
        cases = [(2049, 9, 1.0, 1 << 18, 2, None, REF), (2049, 9, 1.0, 1 << 18, 2, None, FAST)]
    else:
        check_rejections(comm)
    for m, L, eps, min_rows, nu, fuse, arith in cases:
        run_case(comm, rank, world, m, L, eps, min_rows, nu, fuse, arith, oracle=m <= 513)
    dist.barrier()
    del comm
    dist.destroy_process_group()
    if rank == 0:
        print("SHARDED 2D PARITY OK", flush=True)


if __name__ == "__main__":
    main()
