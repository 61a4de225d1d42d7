"""The reference's Optimizer-level tests against the C++ host mirror (include/mppi_optimizer.hpp): tests/cpp/test_optimizer.cpp
is compiled against the CPU oracle here (host logic: setOffset, fallback, twist index, shift, smoke) and against the
CUDA library on the GPU box.  The executables go to a temporary directory: the checkout may be read-only."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "cpp", "test_optimizer.cpp")


@pytest.fixture(scope="module")
def out_dir(tmp_path_factory):
    return str(tmp_path_factory.mktemp("cpp_build"))


def _build(out_dir, name, libdir, lib, defines):
    exe = os.path.join(out_dir, name)
    cmd = ["g++", "-std=c++17", "-O1", "-Wall", "-I", os.path.join(ROOT, "include"), *defines, SRC, "-o", exe,
           "-L", libdir, "-l" + lib, "-Wl,-rpath," + libdir]
    subprocess.run(cmd, check=True)
    return exe


def test_host_mirror_against_oracle(oracle_fns, out_dir):
    exe = _build(out_dir, "test_optimizer_oracle", os.path.join(ROOT, "oracle", "_build"), "mppi_oracle",
                 ["-DMPPI_ABI_PREFIX=oracle_", "-DMPPI_ABI_DECLARE_PREFIXED"])
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr


@pytest.mark.gpu
def test_host_mirror_against_cuda_library(product_fns, out_dir):
    exe = _build(out_dir, "test_optimizer_cuda", os.path.join(ROOT, "mpcholonavigation_b200"), "mppi_b200", [])
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr


# ---- the compiled plugin shim (shim/): sortham::Optimizer + CriticManager + 12 critics over libmppi_b200.so ----------------
SHIM = os.path.join(ROOT, "shim")


def _build_shim(out_dir):
    exe = os.path.join(out_dir, "test_shim")
    libdir, odir = os.path.join(ROOT, "mpcholonavigation_b200"), os.path.join(ROOT, "oracle", "_build")
    cmd = ["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-Wno-unused-parameter",
           "-I", os.path.join(SHIM, "fake_ros"), "-I", os.path.join(SHIM, "include"), "-I", os.path.join(ROOT, "include"),
           os.path.join(ROOT, "tests", "cpp", "test_shim.cpp"), os.path.join(SHIM, "src", "critics.cpp"),
           os.path.join(SHIM, "src", "critic_manager.cpp"), os.path.join(SHIM, "src", "optimizer.cpp"), "-o", exe,
           "-L", libdir, "-lmppi_b200", "-L", odir, "-lmppi_oracle", "-Wl,-rpath," + libdir, "-Wl,-rpath," + odir]
    subprocess.run(cmd, check=True)
    return exe


def test_shim_compiles_and_configures_from_the_deployed_yaml(oracle_fns, out_dir):
    """no device needed: parameters declared and read (dead keys ignored), the critic table, the robot description"""
    r = subprocess.run([_build_shim(out_dir), "describe"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr


@pytest.mark.gpu
def test_shim_cycles_against_the_oracle(oracle_fns, product_fns, out_dir):
    r = subprocess.run([_build_shim(out_dir), "cycles"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
