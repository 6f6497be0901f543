"""Line-block sharded bilinear 2-D V-cycle on >= 2 GPUs of one node: every level's iterate is
bit-identical to the single-GPU 2-D hierarchy, and rank 0 matches the 2-D oracle.  Each world is
skipped when the node has fewer GPUs."""
import importlib
import os
import subprocess
import sys

import pytest

amg = importlib.import_module("algebraic-multigrid_b200")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def launch(world, halo, port, *args):
    if amg.device_count() < world:
        pytest.skip("needs %d GPUs" % world)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
           "--master-addr", "127.0.0.1", "--master-port", str(port),
           os.path.join(ROOT, "tests", "sharded2d_worker.py"), *args]
    env = dict(os.environ, AMGB_HALO=halo)
    out = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=1200, env=env)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert "SHARDED 2D PARITY OK" in out.stdout


@pytest.mark.gpu
@pytest.mark.parametrize("halo", ["peer", "nccl"])
@pytest.mark.parametrize("world", [2, 4, 8])
def test_sharded_2d_vcycle_matches_single_gpu(world, halo):
    """peer: stand-alone peer-memory exchange kernels; nccl: grouped send/recv."""
    launch(world, halo, 29641 + world + (10 if halo == "nccl" else 0))


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 4, 8])
def test_sharded_2d_vcycle_2049(world):
    launch(world, "peer", 29671 + world, "big")
