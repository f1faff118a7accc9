"""rcn::RCN::evaluate_images (include/rcn.hpp) compiled with g++ as a separate program, tests/cpp/eval_test.cpp: on the GPU
it must agree with the hit rule and cost computed on the host from the library's forward pass.
`cpu` mode needs no GPU: with the devices hidden the model cannot be created (RCN_ERR_CUDA, no CPU fallback)."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "cpp", "eval_test.cpp")
LIB_DIR = os.path.join(ROOT, "mercer_research_b200")


@pytest.fixture(scope="module")
def eval_test(built_library, tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("cpp_eval") / "eval_test")
    cmd = ["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-I", os.path.join(ROOT, "include"), SRC,
           "-L", LIB_DIR, "-lrcn_cuda", "-Wl,-rpath," + LIB_DIR, "-o", exe]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return exe


def run(exe, mode, env=None):
    r = subprocess.run([exe, mode], capture_output=True, text=True, timeout=300, env=env)
    assert r.returncode == 0 and f"{mode} ok" in r.stdout, r.stdout + r.stderr
    return r.stdout


def test_cpp_evaluate_without_a_device_fails_with_cuda_error(eval_test):
    run(eval_test, "cpu", env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))


@pytest.mark.gpu
def test_cpp_evaluate_agrees_with_classify(eval_test):
    run(eval_test, "gpu")
