"""The C++ host side above the C ABI (include/rcn.hpp, mirroring rcn's public API) compiled with g++ and run as a
separate program: tests/cpp/host_test.cpp restates the reference crate's own unit tests (kernel.rs:352-441,
rcn.rs:525-538) and the Appendix-B known answers. `cpu` mode needs no GPU."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "cpp", "host_test.cpp")
LIB_DIR = os.path.join(ROOT, "mercer_research_b200")


@pytest.fixture(scope="module")
def host_test(built_library, tmp_path_factory):
    # built in pytest's temporary directory: the suite also runs from a checkout it cannot write to
    exe = str(tmp_path_factory.mktemp("cpp_host") / "host_test")
    cmd = ["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-I", os.path.join(ROOT, "include"), SRC,
           "-L", LIB_DIR, "-lrcn_cuda", "-Wl,-rpath," + LIB_DIR, "-o", exe]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return exe


def run(exe, mode, *args, env=None):
    r = subprocess.run([exe, mode, *args], capture_output=True, text=True, timeout=300, env=env)
    assert r.returncode == 0 and f"{mode} ok" in r.stdout, r.stdout + r.stderr
    return r.stdout


def test_cpp_host_cpu(host_test, tmp_path):
    """Reference unit tests that need no compute, the contract violations (reported before any device work, with the
    reference's panic classes as status codes) and the no-CPU-fallback rule, through the C++ mirror. The devices are
    hidden, so that the no-fallback rule is checked on a GPU machine too."""
    out = run(host_test, "cpu", str(tmp_path), env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert "a CUDA device is present" not in out, "the devices were not hidden: the no-CPU-fallback check did not run\n" + out


@pytest.mark.gpu
def test_cpp_host_gpu(host_test):
    """convolve_2d_padding_same, the Appendix-B Sobel / pooling / argmax / MLP-step known answers, weight_init's shape and
    a seeded RCN::train run (bit-identical when repeated) through the C++ mirror on cuda:0."""
    run(host_test, "gpu")
