"""Worker of tests/test_gpu_gmres.py (launched with torch.distributed.run, one rank per GPU): on a line-block
sharded bilinear 2-D hierarchy, amgb_solve_gmres is rejected with AMGB_ESTATE on every rank, and the
hierarchy still cycles afterwards."""
import importlib
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
amg = importlib.import_module("algebraic-multigrid_b200")


def id_exchanger(raw):
    box = [raw]
    dist.broadcast_object_list(box, src=0)
    return box[0]


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(rank)
    dist.init_process_group("gloo")
    comm = amg.Comm(rank, world, id_exchanger)
    m, L = 129, 6
    A, b = amg.Grid.laplacian(m), amg.Grid.rhs(m)
    mg = amg.Multigrid(amg.BilinearInterpolator2D(L), amg.DampedJacobi(2.0 / 3.0, 2), A, b, L, 1e-9, 1, 1,
                       comm=comm, min_rows_per_rank=1024)
    assert mg.n_sharded_levels() >= 1
    try:
        mg.solve_gmres(1e-8)
    except amg.AmgbError as e:
        assert e.code == amg.ESTATE and "single GPU" in str(e), e
    else:
        raise AssertionError("solve_gmres ran on a sharded hierarchy")
    mg.vcycle()
    mg.get_soln(0)  # collective
    del mg
    dist.barrier()
    if rank == 0:
        print("GMRES SHARDED REJECTED OK", flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
