"""The windowed bilinear 2-D transfer kernels on one GPU: a block of lines addressed through shifted
pointers (as a rank of a sharded level addresses its block) gives the bits of the whole-level call
on the window and touches nothing outside it (tests/cuda/transfer2d_window.cu, built with nvcc for
sm_100a into a temporary directory)."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def exe(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("transfer2d") / "transfer2d_window")
    subprocess.check_call(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17",
                           "-Xcompiler", "-ffp-contract=off",
                           "-I", os.path.join(ROOT, "algebraic-multigrid_b200", "csrc"),
                           os.path.join(ROOT, "tests", "cuda", "transfer2d_window.cu"), "-o", out])
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("m", [64, 65, 257, 300])
def test_windowed_transfers_match_whole_level(exe, m):
    r = subprocess.run([exe, str(m)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.startswith("OK"), r.stdout + r.stderr
