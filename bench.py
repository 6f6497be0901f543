#!/usr/bin/env python
"""bench.py -- throughput of the B200-native multigrid V-cycle path.  Prints ONE JSON line.

Workloads (BASELINE.json configs; SURVEY.md section 8d):
  vcycle4097 (default, configs[2], the headline): 2-D five-point Poisson, 4097x4097 interior
      grid, fp64, 18 levels (coarsest 127 DOF), damped Jacobi (omega 2/3, 2 pre + 2 post sweeps),
      device-resident V-cycles replayed as a CUDA graph; row-block sharded for --gpus > 1.
  gs1025     (configs[1]): 1025x1025, the reference's symmetric Gauss-Seidel smoother, 1 GPU.
  aniso4097  (configs[4]): 4097x4097 anisotropic diffusion, eps = 1e-3 on the +-n coupling.
  micro8193  (configs[3]): one Jacobi sweep, one colour-complete multicolour sweep and one
      residual on the 8193x8193 five-point operator (67 M rows, 335 M entries), halo exchange
      included on >1 GPU.
One "step" is one V-cycle (micro8193: one Jacobi sweep).

Every line carries `parity`: the same cycles from a zero guess on the GPU and in the CPU oracle,
relative differences of the level-0 iterate and of sum r^2 (contract: <= 1e-12, north star).  A
line whose parity fails exits 1.

  python bench.py --gpus 1 --steps 20 --warmup 3
  python bench.py --impl reference ...   # the reference algorithm on host cores
  python bench.py --dump-outputs DIR ... # also write the computed arrays as DIR/<name>.npy

`--dump-outputs DIR` writes, in float64, what the timed path hands its caller: the level-0 iterate
after the last timed V-cycle (`u_level0`); for micro8193, one damped-Jacobi sweep (`jacobi_sweep`)
and one residual (`residual`) of the start iterate the timed launches work on.  A vector longer than
2^21 entries is cut to a fixed, seeded sample of 2^21 of them (16 MB).  The inputs depend only on
the arguments, so two builds run with the same arguments can be compared array for array.

`--impl reference` times the reference's own V-cycle (symmetric Gauss-Seidel,
/root/reference/include/amg/multigrid.hpp:263-305) as restated by the CPU oracle -- the
reference cannot be compiled here (Eigen 3.4.0 absent) -- on the same grid, single-threaded
like the reference.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the tree may be read-only: leave no __pycache__ in it

WORKLOADS = {
    "vcycle4097": dict(n=4097, eps=1.0, smoother="jacobi"),
    "gs1025": dict(n=1025, eps=1.0, smoother="gs"),
    "aniso4097": dict(n=4097, eps=1e-3, smoother="jacobi"),
    "micro8193": dict(n=8193, eps=1.0, smoother="jacobi"),
}
PARITY_TOL = 1e-12   # north star: iterates and residual norms within 1e-12 relative


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=100)
    p.add_argument("--warmup", type=int, default=5)
    p.add_argument("--impl", default="b200", choices=["b200", "reference"])
    p.add_argument("--workload", default="vcycle4097", choices=sorted(WORKLOADS))
    p.add_argument("--n", type=int, default=0, help="override the workload's interior grid points per direction")
    p.add_argument("--levels", type=int, default=0, help="0 = coarsen until <= 200 DOF")
    p.add_argument("--smoother", default="", choices=["", "jacobi", "color", "gs"])
    p.add_argument("--eps", type=float, default=0.0, help="override the anisotropy of the +-n coupling")
    p.add_argument("--arith", default="fast", choices=["fast", "reference"],
                   help="damped-Jacobi kernels: 'fast' = FMA + refined reciprocal (<= 1e-12 vs the oracle, "
                        "checked by the parity leg); 'reference' = the oracle's operation order, bit-identical")
    p.add_argument("--min-rows-per-rank", type=int, default=1 << 17,
                   help="levels with fewer rows per rank are agglomerated (replicated) instead of sharded")
    p.add_argument("--compress", action="store_true",
                   help="opt-in compressed operator formats: matrix-free legs where the operator is verified to be a "
                        "constant five-point stencil, row-type dictionary legs where it has <= 256 distinct rows")
    p.add_argument("--parity-cycles", type=int, default=3)
    p.add_argument("--no-parity", action="store_true")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--dump-outputs", metavar="DIR", default="",
                   help="write the arrays the timed path computed in its last step as DIR/<name>.npy")
    a = p.parse_args()
    if a.steps < 1:
        p.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        p.error("--dump-outputs writes the outputs of the GPU path (--impl b200)")
    if a.dump_outputs and a.workload == "micro8193" and int(os.environ.get("WORLD_SIZE", "1")) > 1:
        p.error("--dump-outputs: micro8193 writes its outputs on one GPU only")
    w = WORKLOADS[a.workload]
    a.n = a.n or w["n"]
    a.eps = a.eps or w["eps"]
    a.smoother = a.smoother or w["smoother"]
    return a


def default_levels(amg, n):
    """Coarsen with the reference's size rule (multigrid.hpp:127-130) until <= 200 DOF."""
    sizes = [n * n]
    while sizes[-1] > 200:
        sizes.append(amg.lib().amgb_n_H_dofs_from_n_h_dofs(sizes[-1]))
    return len(sizes)


def workload_name(a):
    """Same string for both arms: the problem and the operation; the smoother is a separate
    config key (the reference only has symmetric Gauss-Seidel)."""
    if a.workload == "micro8193":
        return "poisson2d_%dx%d_fp64_sweep_residual_microbench" % (a.n, a.n)
    return "poisson2d_%dx%d_fp64_vcycle%s" % (a.n, a.n, "" if a.eps == 1.0 else "_eps%g" % a.eps)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons while the timed region runs."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        import datetime
        for line in self.proc.stdout:
            cells = [c.strip() for c in line.split(",")]
            try:   # nvidia-smi's own wall-clock stamp (the pipe may deliver lines late)
                at = datetime.datetime.strptime(cells[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
            except (ValueError, IndexError):
                at = time.time()
            self.rows.append([at] + cells[1:])

    def stop(self, t0=None, t1=None):
        """Median SM clock / throttle reasons of the samples that arrived in [t0, t1] (the timed
        region); nvidia-smi is started long before it because it needs about a second to come up."""
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = [r[1:] for r in self.rows if t0 is None or t0 <= r[0] <= t1 + 0.05]
        window = "timed region"
        if not rows:   # region shorter than the sampling period: the samples right around it
            near = [r[1:] for r in self.rows if t0 - 0.25 <= r[0] <= t1 + 0.25] if t0 is not None else []
            rows = near or [r[1:] for r in self.rows[-3:]]
            window = "+-0.25 s around the timed region (it is shorter than the sampling period)"
        for r in rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for k, nm in enumerate(names):
                if len(r) > 3 + k and r[3 + k].lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None,
                "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "window": window, "reasons": sorted(reasons)}


DUMP_SAMPLE = 1 << 21


def dump_outputs(d, arrays):
    """Write every array as d/<name>.npy in float64; one longer than DUMP_SAMPLE entries is cut to
    the entries at DUMP_SAMPLE indices drawn with a fixed seed (the same indices for the same size)."""
    import numpy as np
    os.makedirs(d, exist_ok=True)
    for name, x in arrays.items():
        x = np.asarray(x, np.float64).reshape(-1)
        if x.size > DUMP_SAMPLE:
            x = x[np.sort(np.random.default_rng(0).choice(x.size, DUMP_SAMPLE, replace=False))]
        np.save(os.path.join(d, name + ".npy"), x)


def measured_hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(key, world):
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture
    (profiles/traffic.json), 1-GPU launches only: on a sharded run a rank's launch covers 1/world of
    the rows and no capture of it exists, so the key is null there."""
    if world != 1:
        return None
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f).get(key)
    except Exception:
        return None


# ------------------------------------------------------------------------------------------
# CPU oracle legs (rank 0 only): parity checker and the reference-algorithm timing.  The oracle is
# test infrastructure; it is imported here and nowhere in the product.
# ------------------------------------------------------------------------------------------
class OracleSide:
    def __init__(self, a, levels, b):
        global np
        import numpy as np
        import oracle as O
        self.O = O
        t0 = time.perf_counter()
        self.mg = O.Multigrid(O.laplacian(a.n, a.eps), b, levels, 1e-9, 1, 1, O.SMOOTHER_GS, 1, 2.0 / 3.0)
        self.setup_s = time.perf_counter() - t0

    def cycles_from_zero(self, kind, iters, omega, cycles):
        self.mg.set_smoother(kind, iters, omega)
        self.mg.reset()
        for _ in range(cycles):
            self.mg.vcycle()
        u = self.mg.u(0).copy()
        # sum r^2 twice: the reference's sequential sum (common.hpp:22-25) and an accurate (pairwise,
        # numpy) sum of the same residual vector.  Over 1.7e7 terms the sequential sum itself carries
        # ~1e-11 relative rounding, more than the 1e-12 contract, so the GPU's tree sum is compared
        # with the accurate one; both are reported.
        r = self.O.residual(self.mg.A(0), u, self.mg.f(0))
        return u, float(np.dot(r, r)), self.mg.rss()

    def time_reference_vcycles(self, steps, warmup):
        """The reference algorithm (symmetric Gauss-Seidel V-cycle) on one host core."""
        self.mg.set_smoother(self.O.SMOOTHER_GS, 1, 2.0 / 3.0)
        self.mg.reset()
        for _ in range(warmup):
            self.mg.vcycle()
        t0 = time.perf_counter()
        for _ in range(steps):
            self.mg.vcycle()
        dt = time.perf_counter() - t0
        return steps / dt, dt / steps


def bounded_cpu_steps(a, want, budget_s):
    per = 3.3 * (a.n / 4097.0) ** 2   # one symmetric-GS V-cycle of the oracle on one core
    return max(1, min(want, int(budget_s / per) or 1)), per


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import numpy as np
    import oracle as O
    if a.workload == "micro8193":
        return run_reference_micro(a)
    sizes = [a.n * a.n]
    while sizes[-1] > 200:
        sizes.append(O.n_H_from_n_h(sizes[-1]))
    levels = a.levels or len(sizes)
    steps, per = bounded_cpu_steps(a, a.steps, 30.0)
    warm = 1 if per < 10 else 0
    side = OracleSide(a, levels, O.rhs(a.n))
    vps, sec = side.time_reference_vcycles(steps, warm)
    out = {
        "impl": "reference", "metric": "vcycles_per_s", "value": vps, "unit": "V-cycles/s",
        "n_gpus": a.gpus, "steps": steps, "warmup": warm, "ms_per_step": sec * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": workload_name(a), "n": a.n, "levels": levels,
                   "smoother": "symmetric Gauss-Seidel x1 (reference default)",
                   "mdof_per_s": vps * a.n * a.n / 1e6, "setup_s": side.setup_s},
        "cpu_baseline": {"value": vps, "unit": "V-cycles/s", "cores": 1, "kind": "port",
                         "sample": "%d full V-cycle(s) of the oracle restatement of the reference "
                                   "(Eigen absent => reference not compilable), setup excluded, "
                                   "single-threaded like the reference" % steps},
        "e2e": {"value": vps, "unit": "V-cycles/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(out))


def run_reference_micro(a):
    """Reference arm of the microbench: one forward Gauss-Seidel direction (the reference's
    smoother pass, smoother.hpp:148-157) of the oracle on the same operator, one core."""
    import numpy as np
    import oracle as O
    A, b = O.laplacian(a.n, a.eps), O.rhs(a.n)
    u = np.zeros_like(b)
    steps = max(1, min(a.steps, 6))
    O.gs_forward(A, b, u)
    t0 = time.perf_counter()
    for _ in range(steps):
        O.gs_forward(A, b, u)
    dt = (time.perf_counter() - t0) / steps
    print(json.dumps({
        "impl": "reference", "metric": "sweeps_per_s", "value": 1.0 / dt, "unit": "sweeps/s",
        "n_gpus": a.gpus, "steps": steps, "warmup": 1, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(a), "n": a.n,
                   "smoother": "one forward Gauss-Seidel direction (reference smoother pass)"},
        "cpu_baseline": {"value": 1.0 / dt, "unit": "sweeps/s", "cores": 1, "kind": "port",
                         "sample": "%d forward Gauss-Seidel directions of the oracle over the whole %dx%d operator"
                                   % (steps, a.n, a.n)},
        "e2e": {"value": 1.0 / dt, "unit": "sweeps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


# ------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------
def init_dist(amg, a):
    import torch
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    amg.lib().amgb_set_device(local)
    dist = comm = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

        def exchange_id(raw):
            box = [raw]
            dist.broadcast_object_list(box, src=0, device=torch.device("cuda", local))
            return box[0]
        comm = amg.Comm(rank, world, exchange_id)
    return rank, world, local, dist, comm


def run_b200(a):
    import numpy as np
    import torch
    amg = importlib.import_module("algebraic-multigrid_b200")
    # Libraries (NCCL's version banner, ...) write to the C-level stdout: route everything but
    # the final JSON line to stderr
    json_fd = os.dup(1)
    os.dup2(2, 1)
    rank, world, local, dist, comm = init_dist(amg, a)
    if world > 1 and a.smoother == "gs":
        raise SystemExit("lexicographic Gauss-Seidel is a single-GPU path (global dependency chain)")
    if a.workload == "micro8193":
        return run_micro(a, amg, rank, world, local, dist, comm, json_fd)

    levels = a.levels or default_levels(amg, a.n)
    smoother = {"jacobi": amg.DampedJacobi(2.0 / 3.0, 2), "color": amg.MulticolorGaussSeidel(1),
                "gs": amg.SparseGaussSeidel()}[a.smoother]
    arith = amg.ARITH_FAST if (a.arith == "fast" and a.smoother == "jacobi") else amg.ARITH_REFERENCE
    sampler = ClockSampler(local) if rank == 0 else None   # running well before the timed region
    t0 = time.perf_counter()
    A = amg.Grid.laplacian(a.n, a.eps)
    b = amg.Grid.rhs(a.n)
    generate_s = time.perf_counter() - t0
    fuse = (1 | 4 | 16 | 32 | 64 | 128) if a.compress else None
    # one throw-away 35x35 hierarchy first: CUDA context, module load and kernel attributes are
    # process start-up, not hierarchy setup
    warm = amg.Multigrid(None, smoother, amg.Grid.laplacian(35), amg.Grid.rhs(35), 8, 1e-9, 1, 1)
    warm.vcycle()
    warm.synchronize()
    del warm
    t0 = time.perf_counter()
    mg = amg.Multigrid(None, smoother, A, b, levels, 1e-9, 1, 1, comm=comm,
                       min_rows_per_rank=a.min_rows_per_rank, arith=arith, fuse=fuse)
    setup_s = time.perf_counter() - t0
    N0 = mg.get_n_dofs(0)

    stream = torch.cuda.Stream()
    mg.set_stream(stream.cuda_stream)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if dist is None:
            return x
        t = torch.tensor([x], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident V-cycles (value) ----
    n_warm = max(a.warmup, 3)   # timing rule: at least three untimed cycles (graph built, clocks up)
    for _ in range(n_warm):
        mg.vcycle()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = amg.kernel_launches()
    tw0 = time.time()
    e0.record(stream)
    for _ in range(a.steps):
        mg.vcycle()
    e1.record(stream)
    barrier()
    tw1 = time.time()
    ms = max_over_ranks(e0.elapsed_time(e1))
    launches = amg.kernel_launches() - launches0
    clocks = sampler.stop(tw0, tw1) if sampler else None
    # one problem, row blocks spread over the ranks: whole-job V-cycles = steps
    vps = a.steps / (ms * 1e-3)
    rss_after = mg.rss()
    if a.dump_outputs:
        u_last = mg.get_soln(0)    # collective on >1 GPU: every rank takes part
        if rank == 0:
            dump_outputs(a.dump_outputs, {"u_level0": u_last})
        del u_last

    # ---- e2e: host-resident b and u; H2D(b,u) + V-cycle + D2H(u) each step, through the C ABI.
    # On >1 GPU every rank owns the row block [r0, r1) of b and u (amgb_hierarchy_*_local): the
    # job moves the same 24 N0 bytes per step, 1/world of them per rank and PCIe link. ----
    e2e = None
    r0, r1 = mg.local_range(0)
    if not a.no_e2e:
        nloc = (r1 - r0) if world > 1 else N0
        hb = torch.from_numpy(np.ascontiguousarray(b[r0:r1] if world > 1 else b)).pin_memory()
        hu = torch.zeros(nloc, dtype=torch.float64).pin_memory()
        steps_e = max(3, min(a.steps, 10))

        def e2e_step():
            if world > 1:
                mg.set_rhs_local(0, hb.numpy()); mg.set_soln_local(0, hu.numpy())
                mg.vcycle()
                mg.get_soln_local(0, hu.numpy())     # synchronises
            else:
                mg.set_rhs(0, hb.numpy()); mg.set_soln(0, hu.numpy())
                mg.vcycle()
                mg.get_soln(0, hu.numpy())           # synchronises
        for _ in range(2):
            e2e_step()
        barrier()
        t1 = time.perf_counter()
        for _ in range(steps_e):
            e2e_step()
        barrier()
        dt = max_over_ranks(time.perf_counter() - t1)
        e2e = {"value": steps_e / dt, "unit": "V-cycles/s",
               "h2d_bytes_per_step": 16 * N0, "d2h_bytes_per_step": 8 * N0, "steps": steps_e,
               "note": "whole-job bytes; each of the %d rank(s) moves its own row block of b, u "
                       "(pinned host memory) through amgb_hierarchy_set_rhs/soln%s and get_soln%s" % (
                           world, "_local" if world > 1 else "", "_local" if world > 1 else "")}

    # ---- parity: the same cycles from the zero guess on the GPU and in the oracle ----
    parity = None
    u_gpu = rss_gpu = None
    if not a.no_parity:
        mg.set_soln(0, np.zeros(N0))
        mg.set_rhs(0, b)
        for _ in range(a.parity_cycles):
            mg.vcycle()
        u_gpu = mg.get_soln(0)     # collective on >1 GPU: every rank takes part
        rss_gpu = mg.rss()

    # ---- dominant kernel roofline, timed live with CUDA events on the handle's stream ----
    # Algorithmic bytes of one pass over level l for the layout the kernel streams
    # (DESIGN.md "bytes per unit"): stored matrix bytes (DIA: 8 B x diagonals x rows, no
    # index array; SELL: 12 B per stored entry) + f read + u read + result write (24 N).
    # The CSR-based figure of SURVEY.md 8(d) (12 nnz + 28 N + 4) is reported beside it.
    peak, peak_src = measured_hbm_peak()
    n1 = mg.get_n_dofs(1)
    survey0 = mg.pass_bytes(0)
    fused0 = mg.fused_legs(0)
    per_kernel = {}

    def mat_bytes(l):
        """operator bytes a leg of level l streams on this rank: none when the level runs matrix-free,
        one byte per row when it runs from a row-type dictionary, else the stored DIA / SELL bytes"""
        if mg.matrix_free(l):
            return 0
        a0, a1 = mg.local_range(l)
        if mg.dictionary_types(l):
            return a1 - a0
        if mg.fused_legs(l) and mg.n_diagonals(l) > 0:
            return 8 * mg.n_diagonals(l) * (a1 - a0)    # a leg streams every diagonal of its rows
        return mg.matrix_bytes(l)

    legs_timed = []
    if fused0:
        # Fused legs (one pass per level and leg).  Algorithmic bytes of a leg on this rank's rows:
        # operator (unless matrix-free) + f + input read + result written (+ coarse rhs / correction);
        # the dominant kernel of the cycle is the slowest of the legs of the three finest levels.
        for l in range(min(3, levels - 1)):
            if not mg.fused_legs(l):
                break
            a0, a1 = mg.local_range(l)
            rows = a1 - a0
            for kind, nm in ((4, "down"), (5, "up")):
                t_ms = mg.time_kernel(l, kind, warmup=3, reps=20)
                alg = mat_bytes(l) + ((24 if (l == 0 or kind == 5) else 16) * rows) + 8 * (rows // 2)
                legs_timed.append({"level": l, "leg": nm, "ms": t_ms, "algorithmic_bytes": alg,
                                   "GB/s": alg / (t_ms * 1e-3) / 1e9, "frac": alg / (t_ms * 1e-3) / 1e9 / peak,
                                   "matrix_free": bool(mg.matrix_free(l)), "dictionary_types": mg.dictionary_types(l)})
        top = max(legs_timed, key=lambda x: x["ms"])
        kern_ms, bytes0 = top["ms"], top["algorithmic_bytes"]
        plan = mg.leg_plan(top["level"], up=(top["leg"] == "up"))
        kname = "k_stream_leg" if plan["smem_bytes"] == 0 else "k_fused_leg"
        traffic_key = "%s_L%d_%s%s" % (kname, top["level"], top["leg"], "_fast" if arith == amg.ARITH_FAST else "")
        kdesc = "%s %s leg of level %d (%s; %s arithmetic, %s)" % (
            kname, top["leg"], top["level"],
            "%d Jacobi sweeps + residual + restriction in one pass" % smoother.n_iters if top["leg"] == "down"
            else "prolongation + add + %d Jacobi sweeps in one pass" % smoother.n_iters,
            "fast" if arith == amg.ARITH_FAST else "reference-order",
            "matrix-free five-point stencil" if top["matrix_free"] else
            "row-type dictionary, %d types" % top["dictionary_types"] if top["dictionary_types"] else
            mg.format(top["level"]) + " layout")
    else:
        kern_ms = mg.time_kernel(0, 0, warmup=3, reps=20)
        bytes0 = mg.matrix_bytes(0) + 24 * (r1 - r0)       # this rank's row block
        plan = None
        gs_name = ("k_gs_wave (one forward direction, multi-SM wavefront)"
                   if a.smoother == "gs" and mg.gs_kernel(0) == amg.GS_KERNEL_WAVE
                   else "k_gs_rhs + k_gs_lines (one forward direction)")
        kname = {"jacobi": "k_jacobi", "color": "k_color_gs (all colours)", "gs": gs_name}[a.smoother]
        traffic_key = kname.split(" ")[0]
        kdesc = kname + " (level 0, %s layout)" % mg.format(0)
    achieved = bytes0 / (kern_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "kernel": kdesc,
                "achieved": achieved, "peak": peak,
                "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": bytes0, "ms_per_launch": kern_ms,
                "survey_formula_bytes_per_launch": survey0,
                "survey_formula_GBps": survey0 / (kern_ms * 1e-3) / 1e9,
                "traffic": ncu_traffic(traffic_key, world)}
    if a.smoother == "gs":
        roofline["note"] = ("lexicographic Gauss-Seidel is bound by its dependency depth, not by HBM "
                            "(SURVEY.md 8d): GB/s is reported for completeness")
    if plan:
        roofline["tiling"] = plan
        roofline["legs"] = legs_timed
    pass0 = mg.matrix_bytes(0) + 24 * (r1 - r0)
    kinds = [(0, "smoother_sweep"), (1, "residual"), (2, "residual_restrict"), (3, "prolong_add")]
    if fused0:
        kinds += [(4, "fused_down_leg"), (5, "fused_up_leg")]
    for kind, nm in kinds if world == 1 else ():
        t_ms = mg.time_kernel(0, kind, warmup=3, reps=20)
        alg = {0: pass0, 1: pass0, 2: mg.matrix_bytes(0) + 16 * N0 + 8 * n1, 3: 8 * n1 + 16 * N0,
               4: mat_bytes(0) + 24 * N0 + 8 * n1, 5: mat_bytes(0) + 24 * N0 + 8 * n1}[kind]
        per_kernel[nm] = {"ms": t_ms, "GB/s": alg / (t_ms * 1e-3) / 1e9,
                          "frac": alg / (t_ms * 1e-3) / 1e9 / peak}
    # bytes one V-cycle must move with the layouts and kernels in use
    passes = 2 * smoother.n_iters if a.smoother == "jacobi" else 4 * smoother.n_iters
    layout_bytes = 0
    for l in range(levels - 1):
        nl, nn = mg.get_n_dofs(l), mg.get_n_dofs(l + 1)
        if mg.fused_legs(l):
            down = mat_bytes(l) + (24 if l == 0 else 16) * nl + 8 * nn
            up = mat_bytes(l) + 24 * nl + 8 * nn
            layout_bytes += down + up
        else:
            layout_bytes += (passes + 1) * (mg.matrix_bytes(l) + 24 * nl) + 24 * nl + 16 * nn
    vbytes = mg.vcycle_bytes()
    phases = mg.phase_times() if hasattr(mg, "phase_times") else None

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    # ---- rank 0: the CPU oracle legs ----
    cpu = None
    ok = True
    if not (a.no_parity and (a.no_cpu_baseline or world > 1)):
        side = OracleSide(a, levels, b)
        if not a.no_parity:
            kind = {"jacobi": side.O.SMOOTHER_JACOBI, "color": side.O.SMOOTHER_COLOR_GS,
                    "gs": side.O.SMOOTHER_GS}[a.smoother]
            u_cpu, rss_cpu, rss_seq = side.cycles_from_zero(kind, smoother.n_iters, 2.0 / 3.0, a.parity_cycles)
            rel_u = float(np.linalg.norm(u_gpu - u_cpu) / np.linalg.norm(u_cpu))
            rel_rss = abs(rss_gpu - rss_cpu) / rss_cpu
            ok = bool(rel_u <= PARITY_TOL and rel_rss <= PARITY_TOL)
            parity = {"cycles": a.parity_cycles, "from": "zero guess, same b", "rel_u_level0": rel_u,
                      "rel_rss": rel_rss, "rss_gpu": rss_gpu, "rss_oracle": rss_cpu,
                      "rss_oracle_sequential_sum": rss_seq,
                      "rss_note": "rss_oracle = accurate (pairwise) sum of the oracle's residual vector; the reference's "
                                  "sequential sum of the same vector is off by %.1e relative on its own" % (
                                      abs(rss_seq - rss_cpu) / rss_cpu),
                      "tol": PARITY_TOL, "ok": ok,
                      "bit_identical_u": bool(u_gpu.tobytes() == u_cpu.tobytes()), "n_gpus": world}
        if not a.no_cpu_baseline and world == 1:   # contract: the CPU baseline is timed at N = 1 only
            cs, _ = bounded_cpu_steps(a, 5, 12.0)
            cvps, _ = side.time_reference_vcycles(cs, 0)
            cpu = {"value": cvps, "unit": "V-cycles/s", "cores": 1, "kind": "port",
                   "host_cores_available": os.cpu_count(),
                   "sample": "%d full reference V-cycle(s) (symmetric Gauss-Seidel, the reference's "
                             "smoother) of the oracle on the same %dx%d grid, setup excluded; the "
                             "reference is single-threaded by construction" % (cs, a.n, a.n)}

    out = {
        "metric": "vcycles_per_s", "value": vps, "unit": "V-cycles/s", "n_gpus": world,
        "steps": a.steps, "warmup": n_warm, "ms_per_step": ms / a.steps,
        "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(a), "n": a.n, "n_dofs": N0, "levels": levels,
                   "smoother": a.smoother, "smoother_iters": smoother.n_iters,
                   "omega": getattr(smoother, "omega", None),
                   "arith": "fast (FMA, refined reciprocal)" if arith == amg.ARITH_FAST else "reference order",
                   "operator_formats": "compressed where verified (matrix-free / row-type dictionary legs)" if a.compress
                                       else "general (DIA rows streamed from HBM)",
                   "l2_policy": "inputs larger than L2 (level-0 operator+vectors stream %.2f GB per "
                                "pass, L2 is 126 MB)" % (bytes0 / 1e9) if bytes0 > 3e8 else
                                "level-0 pass streams %.0f MB: L2-resident, reported as such" % (bytes0 / 1e6),
                   "parallelism": "single GPU" if world == 1 else
                                  "row blocks x%d, %d sharded levels, halo via %s (%d stand-alone exchange launches "
                                  "per V-cycle), coarser levels replicated after one gather" % (
                                      world, mg.n_sharded_levels(),
                                      {"peer": "peer-memory stores over NVLink + epoch flags",
                                       "nccl": "NCCL send/recv"}.get(mg.halo_mode(), mg.halo_mode()),
                                      mg.halo_exchanges_per_vcycle()),
                   "mdof_per_s": vps * N0 / 1e6, "setup_s": setup_s, "generate_s": generate_s,
                   "rss_after_timed_cycles": rss_after,
                   "fused_legs": [bool(mg.fused_legs(l)) for l in range(levels - 1)], "tail_first": mg.tail_first(),
                   "matrix_free_levels": [l for l in range(levels - 1) if mg.matrix_free(l)],
                   "dictionary_types": [mg.dictionary_types(l) for l in range(levels - 1)],
                   "mid_levels": list(mg.mid_range()),
                   "launches_per_vcycle": mg.launches_per_vcycle(),
                   "vcycle_layout_bytes": layout_bytes,
                   "vcycle_hbm_frac": (layout_bytes / (ms / a.steps * 1e-3) / 1e9 / peak) if world == 1 else None,
                   "vcycle_survey_formula_bytes": vbytes,
                   "layouts": [mg.format(l) for l in range(levels)],
                   "gs_kernels": ([{0: "fronts", 1: "linescan", 2: "wavefront"}.get(mg.gs_kernel(l)) for l in range(levels - 1)]
                                  if a.smoother == "gs" else None),
                   "kernels_level0": per_kernel, "phases_ms": phases},
        "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "parity": parity,
        "gpu_launches": launches, "clocks": clocks,
    }
    os.write(json_fd, (json.dumps(out) + "\n").encode())
    if dist is not None:
        dist.destroy_process_group()
    if not ok:
        sys.stderr.write("PARITY FAILED: %r\n" % (parity,))
        sys.exit(1)


def run_micro(a, amg, rank, world, local, dist, comm, json_fd):
    """configs[3]: sweeps/s and GB/s of one damped-Jacobi sweep and one residual on the 8193^2 five-point
    operator -- on >1 GPU each rank sweeps its row block and the halo exchange with ranks +-1 is inside
    the timed launches -- plus one colour-complete multicolour Gauss-Seidel sweep (1 GPU).  The operator
    is level 0 of an ordinary hierarchy (device-side setup); parity: one sweep and one residual of the
    whole 67 M-row level against the oracle's arithmetic (oracle.five_point_*), bit for bit."""
    import numpy as np
    import torch
    sampler = ClockSampler(local) if rank == 0 else None
    t0 = time.perf_counter()
    A = amg.Grid.laplacian(a.n, a.eps)
    b = amg.Grid.rhs(a.n)
    generate_s = time.perf_counter() - t0
    levels = a.levels or default_levels(amg, a.n)
    omega = 2.0 / 3.0
    t0 = time.perf_counter()
    mg = amg.Multigrid(None, amg.DampedJacobi(omega, 1), A, b, levels, 1e-9, 1, 1, comm=comm,
                       min_rows_per_rank=a.min_rows_per_rank, arith=amg.ARITH_REFERENCE)
    setup_s = time.perf_counter() - t0
    N, nnz = a.n * a.n, A.nnz
    stream = torch.cuda.Stream()
    mg.set_stream(stream.cuda_stream)
    u0 = 1e-3 * b + 1.0            # deterministic, non-constant start
    mg.set_soln(0, u0)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if dist is None:
            return x
        t = torch.tensor([x], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    peak, peak_src = measured_hbm_peak()
    n_warm = max(a.warmup, 3)
    r0, r1 = mg.local_range(0)
    launches0 = amg.kernel_launches()
    barrier()
    tw0 = time.time()
    ms_j = max_over_ranks(mg.time_kernel(0, 9, warmup=n_warm, reps=a.steps))     # CUDA events around `steps` launches
    barrier()
    tw1 = time.time()
    ms_r = max_over_ranks(mg.time_kernel(0, 11, warmup=n_warm, reps=a.steps))
    barrier()
    # (the sampler is stopped only now: stopping it takes rank 0 up to a second, and a rank that enters
    # the next collective timing loop late shows up in every other rank's first launches)
    clocks = sampler.stop(tw0, tw1) if sampler else None
    launches = amg.kernel_launches() - launches0
    B0 = 12 * nnz + 28 * N + 4                          # SURVEY.md 8(d): CSR-equivalent bytes per pass
    dia_rank = mg.matrix_bytes(0) + 24 * (r1 - r0)      # what this rank's DIA kernels stream per pass
    kernels = {}
    for nm, ms in (("jacobi_sweep", ms_j), ("residual", ms_r)):
        kernels[nm] = {"ms": ms, "per_s": 1e3 / ms, "layout_bytes_per_gpu": dia_rank,
                       "GB/s_per_gpu": dia_rank / (ms * 1e-3) / 1e9, "frac": dia_rank / (ms * 1e-3) / 1e9 / peak,
                       "survey_formula_GB/s_per_gpu": B0 / world / (ms * 1e-3) / 1e9,
                       "halo_exchange_included": world > 1}
    # ---- parity: one sweep (and, on one GPU, one residual) of the whole level vs the oracle's arithmetic
    import oracle as O
    mg.set_soln(0, u0)
    mg.smooth_level(0)                                   # one damped-Jacobi sweep, halo exchange included
    got = mg.get_soln_local(0) if world > 1 else mg.get_soln(0)
    want = O.five_point_jacobi(a.n, a.eps, u0, b, omega)[r0:r1] if world > 1 else O.five_point_jacobi(a.n, a.eps, u0, b, omega)
    ok = got.tobytes() == want.tobytes()
    rel_sweep = float(np.linalg.norm(got - want) / np.linalg.norm(want))
    rel_res = None
    if world == 1:
        mg.set_soln(0, u0)
        r_gpu = mg.residual_level(0)
        r_cpu = O.five_point_residual(a.n, a.eps, u0, b)
        rel_res = float(np.linalg.norm(r_gpu - r_cpu) / np.linalg.norm(r_cpu))
        ok = ok and r_gpu.tobytes() == r_cpu.tobytes()
        if a.dump_outputs:
            dump_outputs(a.dump_outputs, {"jacobi_sweep": got, "residual": r_gpu})
    if dist is not None:
        t = torch.tensor([1.0 if ok else 0.0], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        ok = bool(t.item() == 1.0)
    parity = {"what": "one damped-Jacobi sweep%s of the whole %dx%d level vs oracle.five_point_* (the oracle's per-row "
                      "arithmetic, vectorised)" % (" and one residual" if world == 1 else " (every rank its row block)", a.n, a.n),
              "rel_sweep": rel_sweep, "rel_residual": rel_res, "bit_identical": ok, "tol": PARITY_TOL, "ok": ok, "n_gpus": world}
    # ---- colour-complete multicolour Gauss-Seidel sweep: single GPU, amgb_matrix mirror of the same operator
    color = None
    if world == 1:
        del mg
        dm = amg.DeviceMatrix(A)
        dm.residual(u0, b)                                # uploads u and f
        ms_c = dm.time_pass(1, omega, warmup=n_warm, reps=a.steps)
        cbytes = dm.stream_bytes(1) + 24 * N
        color = {"ms": ms_c, "per_s": 1e3 / ms_c, "layout_bytes_per_gpu": cbytes, "GB/s_per_gpu": cbytes / (ms_c * 1e-3) / 1e9,
                 "frac": cbytes / (ms_c * 1e-3) / 1e9 / peak, "colors": dm.coloring()[0],
                 "survey_formula_GB/s_per_gpu": B0 / (ms_c * 1e-3) / 1e9}
        kernels["color_gs_sweep"] = color
    else:
        kernels["color_gs_sweep"] = None   # the sharded hierarchy smooths with damped Jacobi; multicolour GS is single-GPU
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    cpu = None
    if not a.no_cpu_baseline and world == 1:
        ns = 2049   # bounded sample: the same operator family at 2049^2 (1/16 of the rows), one core
        Ao, bo = O.laplacian(ns, a.eps), O.rhs(ns)
        AT = Ao.transpose()
        u = bo.copy()
        reps = 5
        t0 = time.perf_counter()
        for _ in range(reps):
            u = O.jacobi_sweep(AT, u, bo, omega)
        dt = (time.perf_counter() - t0) / reps
        cpu = {"value": 1.0 / (dt * (a.n / ns) ** 2), "unit": "sweeps/s", "cores": 1, "kind": "port",
               "host_cores_available": os.cpu_count(),
               "sample": "%d damped-Jacobi sweeps of the oracle at %dx%d (%.3f s each), scaled by the row ratio "
                         "to %dx%d" % (reps, ns, ns, dt, a.n, a.n)}
    out = {
        "metric": "sweeps_per_s", "value": 1e3 / ms_j, "unit": "sweeps/s", "n_gpus": world,
        "steps": a.steps, "warmup": n_warm, "ms_per_step": ms_j, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(a), "n": a.n, "n_dofs": N, "nnz": nnz, "omega": omega,
                   "survey_formula_bytes_per_pass": B0, "setup_s": setup_s, "generate_s": generate_s,
                   "l2_policy": "inputs larger than L2 (%.2f GB per pass per GPU)" % (dia_rank / 1e9),
                   "parallelism": "single GPU" if world == 1 else
                                  "row blocks x%d, one halo exchange with ranks +-1 per sweep / residual (%s), on a side "
                                  "stream beside the sweep of the block interior" % (world, mg.halo_mode()),
                   "kernels": kernels},
        "roofline": {"bound": "hbm", "kernel": "k_jacobi (one damped-Jacobi sweep, DIA layout%s)" % (
                         ", halo exchange included" if world > 1 else ""),
                     "achieved": kernels["jacobi_sweep"]["GB/s_per_gpu"], "peak": peak, "unit": "GB/s",
                     "frac": kernels["jacobi_sweep"]["frac"], "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": dia_rank, "ms_per_launch": ms_j,
                     "survey_formula_bytes_per_launch": B0 // world,
                     "traffic": ncu_traffic("k_jacobi_8193", world)},
        "cpu_baseline": cpu, "parity": parity,
        "e2e": None, "gpu_launches": launches, "clocks": clocks,
    }
    os.write(json_fd, (json.dumps(out) + "\n").encode())
    if dist is not None:
        dist.destroy_process_group()
    if not ok:
        sys.exit(1)


def main():
    a = parse_args()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)


if __name__ == "__main__":
    main()
