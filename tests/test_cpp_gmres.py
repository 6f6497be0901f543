"""Multigrid::solve_gmres in the C++ mirror headers: compiles against the stand-in types and
against the Eigen shim (CPU), and solves an unsymmetric convection-diffusion problem through the C ABI (GPU)."""
import os
import subprocess
import tempfile

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "algebraic-multigrid_b200")
SRC = os.path.join(ROOT, "tests", "cpp", "gmres_mirror.cpp")


def build(eigen):
    exe = os.path.join(tempfile.mkdtemp(prefix="amgb_gmres_"), "gmres_mirror")
    flags = (["-DAMGB_USE_EIGEN", "-I", os.path.join(ROOT, "tests", "cpp", "eigen_shim")] if eigen
             else ["-DAMGB_NO_EIGEN"])
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-Wall"] + flags + ["-I", os.path.join(ROOT, "include"),
                           SRC, "-o", exe, "-L", PKG, "-lamgb", "-Wl,-rpath," + PKG])
    return exe


def test_mirror_compiles_with_stand_in_types():
    subprocess.check_call([build(eigen=False)])


def test_mirror_compiles_against_the_eigen_shim():
    assert os.path.exists(build(eigen=True))


@pytest.mark.gpu
def test_mirror_solves_convection_diffusion_with_gmres():
    out = subprocess.run([build(eigen=False), "gpu"], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout + out.stderr
