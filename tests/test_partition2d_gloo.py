"""CPU: the line-block partition plan of a sharded bilinear 2-D hierarchy (amgb_partition_plan_2d)
and, over gloo at world size 2 and 3, an emulation of the sharded 2-D V-cycle in which every rank
only ever touches its own block and halos (everything else is NaN), exchanges halos with its
neighbours through torch.distributed and must reproduce the 2-D oracle's damped-Jacobi V-cycle."""
import importlib
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)
import oracle as O  # noqa: E402
import oracle_bilinear2d as O2  # noqa: E402

amg = importlib.import_module("algebraic-multigrid_b200")

OMEGA, SWEEPS = 2.0 / 3.0, 2


def lines(m0, n_levels):
    m = [m0]
    for _ in range(1, n_levels):
        m.append(m[-1] // 2)
    return m


def check_plan(m, world, min_rows):
    ns, starts, lo, hi, gh = amg.partition_plan_2d(m, world, min_rows)
    gl = 0
    for l in range(ns - 1, -1, -1):
        gl = 2 * gl + 1
        assert gh[l] == gl * m[l], (l, gh[l])
        assert lo[l] >= m[l] + 2 and hi[l] >= (gl + 1) * m[l] + 2
        assert m[l] * m[l] // world >= min_rows
    for l in range(ns):
        st = starts[l]
        assert st[0] == 0 and st[world] == m[l] * m[l]
        assert (st % m[l] == 0).all()
        assert (np.diff(st) >= max(lo[l], hi[l])).all(), (l, np.diff(st))
        if l + 1 < ns:
            assert (starts[l + 1][:-1] // m[l + 1] == st[:-1] // m[l] // 2).all()
    if ns:
        assert (starts[0][:-1] // m[0] % (1 << ns) == 0).all()
        assert ns + 1 <= len(m)
    return ns, starts, lo, hi, gh


@pytest.mark.parametrize("world", [2, 3, 4, 5, 8])
@pytest.mark.parametrize("m0,n_levels,min_rows", [(65, 5, 60), (64, 5, 60), (257, 7, 1000), (1000, 8, 5000),
                                                  (4097, 12, 1 << 18), (8193, 12, 1 << 18), (513, 8, 1)])
def test_plan_properties(m0, n_levels, min_rows, world):
    check_plan(lines(m0, n_levels), world, min_rows)


def test_plan_shape_at_4097_on_8_ranks():
    ns, starts, lo, hi, gh = check_plan(lines(4097, 12), 8, 1 << 18)
    assert ns == 2
    assert gh[0] == 3 * 4097 and gh[1] == 2048


def test_plan_shrinks_and_declines():
    m = lines(65, 5)
    assert amg.partition_plan_2d(m, 1, 1)[0] == 0              # one rank: nothing to shard
    assert amg.partition_plan_2d(m, 2, 10 ** 6)[0] == 0        # too small for the threshold
    assert amg.partition_plan_2d(m, 40, 1)[0] == 0             # blocks shorter than their halos
    assert amg.partition_plan_2d(m, 2, 1)[0] == len(m) - 1     # every level but the coarsest
    assert amg.partition_plan_2d(m, 3, 1)[0] == len(m) - 2     # level 3 blocks would be shorter than their halos
    assert amg.partition_plan_2d([8], 2, 1)[0] == 0            # the coarsest level is never sharded


@pytest.mark.parametrize("args", [([], 2, 1), ([65, 32], 0, 1), ([65, 33, 16], 2, 1), ([0], 2, 1),
                                  ([65, 32, 16, 8, 4, 2, 1, 1], 2, 1), ([50000, 25000], 2, 1)])
def test_plan_rejects_bad_arguments(args):
    with pytest.raises(amg.InvalidArgument):
        amg.partition_plan_2d(*args)


def sendrecv(rank, world, vec, lo_send, lo_recv, hi_send, hi_recv):
    """Exchange with rank-1 (lo) and rank+1 (hi); all arguments are slices of vec."""
    reqs, bufs = [], []
    if rank > 0:
        reqs.append(dist.isend(torch.from_numpy(vec[lo_send].copy()), rank - 1))
        t = torch.empty(lo_recv.stop - lo_recv.start, dtype=torch.float64)
        reqs.append(dist.irecv(t, rank - 1)); bufs.append((lo_recv, t))
    if rank + 1 < world:
        reqs.append(dist.isend(torch.from_numpy(vec[hi_send].copy()), rank + 1))
        t = torch.empty(hi_recv.stop - hi_recv.start, dtype=torch.float64)
        reqs.append(dist.irecv(t, rank + 1)); bufs.append((hi_recv, t))
    for r in reqs:
        r.wait()
    for sl, t in bufs:
        vec[sl] = t.numpy()


def poison(v):
    """NaN (= never written) becomes inf, so any product that touches it turns the result non-finite."""
    return np.nan_to_num(v, nan=np.inf)


def worker(rank, world, port, m0, L, min_rows, result):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        b = O.rhs(m0)
        mo = O2.Multigrid(O.laplacian(m0), b, L, 1e-9, 1, 1, O.SMOOTHER_JACOBI, SWEEPS, OMEGA)
        m = mo.m
        mats = [mo.A(l).to_scipy().tocsr() for l in range(L)]
        Rs = [mo.R(l).to_scipy().tocsr() for l in range(L - 1)]
        Ps = [mo.P(l).to_scipy().tocsr() for l in range(L - 1)]
        sizes = [k * k for k in m]
        ns, starts, hlo, hhi, ghost = amg.partition_plan_2d(m, world, min_rows)
        assert ns >= 2, ns
        s = [int(starts[l][rank]) for l in range(ns)]
        e = [int(starts[l][rank + 1]) for l in range(ns)]

        def window(l):  # index range this rank may touch on level l
            return max(0, s[l] - hlo[l]), min(sizes[l], e[l] + hhi[l])

        def top(l):  # end of the own + ghost rows
            return min(sizes[l], e[l] + ghost[l])

        u = [np.full(sizes[l], np.nan) if l < ns else np.zeros(sizes[l]) for l in range(L)]
        f = [np.full(sizes[l], np.nan) if l < ns else np.zeros(sizes[l]) for l in range(L)]
        lo, hi = window(0)
        u[0][lo:hi] = 0.0
        f[0][s[0]:top(0)] = b[s[0]:top(0)]

        def exchange(l, v):
            sendrecv(rank, world, v,
                     slice(s[l], s[l] + hhi[l]), slice(max(0, s[l] - hlo[l]), s[l]),
                     slice(e[l] - hlo[l], e[l]), slice(e[l], min(sizes[l], e[l] + hhi[l])))

        def smooth(l):
            d = mats[l].diagonal()
            for _ in range(SWEEPS):
                if l < ns:
                    exchange(l, u[l])
                    rows = slice(s[l], e[l])
                    new = u[l].copy()
                    new[rows] = u[l][rows] + OMEGA * (f[l][rows] - mats[l][rows] @ poison(u[l])) / d[rows]
                    u[l] = new
                else:
                    u[l] = u[l] + OMEGA * (f[l] - mats[l] @ u[l]) / d

        for l in range(L - 1):
            smooth(l)
            if l < ns:
                exchange(l, u[l])
                r = np.full(sizes[l], np.nan)
                r[s[l]:top(l)] = f[l][s[l]:top(l)] - mats[l][s[l]:top(l)] @ poison(u[l])
                assert np.isfinite(r[s[l]:top(l)]).all(), "residual read u outside block + halos"
                if l + 1 < ns:
                    c0, c1 = s[l + 1], top(l + 1)
                else:   # coarse lines from half the fine block's first line
                    c0 = s[l] // m[l] // 2 * m[l + 1]
                    c1 = e[l] // m[l] // 2 * m[l + 1] if rank + 1 < world else sizes[l + 1]
                fc = Rs[l][c0:c1] @ poison(r)
                assert np.isfinite(fc).all(), "restriction read rows outside block + ghost lines"
                if l + 1 < ns:
                    f[l + 1][c0:c1] = fc
                    lo, hi = window(l + 1)
                    u[l + 1][lo:hi] = 0.0
                else:  # first replicated level: gather the blocks, every rank keeps a replica
                    parts = [None] * world
                    dist.all_gather_object(parts, (c0, fc))
                    got = np.zeros(sizes[l + 1], bool)
                    for c, blk in parts:
                        f[l + 1][c:c + len(blk)] = blk
                        got[c:c + len(blk)] = True
                    assert got.all()
                    u[l + 1][:] = 0.0
            else:
                f[l + 1] = Rs[l] @ (f[l] - mats[l] @ u[l])
                u[l + 1][:] = 0.0
        u[L - 1] = O.Ldlt(mo.A(L - 1)).solve(f[L - 1])
        for l in range(L - 2, -1, -1):
            if l + 1 < ns:
                exchange(l + 1, u[l + 1])
            if l < ns:
                corr = Ps[l][s[l]:e[l]] @ poison(u[l + 1])
                assert np.isfinite(corr).all(), "prolongation read coarse rows outside block + halo"
                u[l][s[l]:e[l]] += corr
            else:
                u[l] = u[l] + Ps[l] @ u[l + 1]
            smooth(l)
        mo.vcycle()
        for l in range(L):
            mine = u[l][s[l]:e[l]] if l < ns else u[l]
            ref = mo.u(l)[s[l]:e[l]] if l < ns else mo.u(l)
            assert np.isfinite(mine).all()
            err = np.linalg.norm(mine - ref) / max(np.linalg.norm(ref), 1e-300)
            assert err <= 1e-12, (l, err)
        result[rank] = ns
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("m0,L,min_rows", [(65, 5, 60), (64, 5, 60)])
@pytest.mark.parametrize("world", [2, 3])
def test_emulated_sharded_2d_vcycle(world, m0, L, min_rows):
    mgr = mp.Manager()
    result = mgr.dict()
    mp.spawn(worker, args=(world, 29660 + 4 * world + (m0 & 1), m0, L, min_rows, result), nprocs=world, join=True)
    assert sorted(result.keys()) == list(range(world))
