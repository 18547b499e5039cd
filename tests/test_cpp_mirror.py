"""The C++ host mirror (include/aurora_codecs.hpp) compiles against the C ABI; without a GPU it fails loudly
(CPU test), with one it round-trips the reference's test shapes (GPU test)."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "auroralib", "compression_b200")


@pytest.fixture(scope="module")
def mirror_exe(tmp_path_factory):
    # the executable goes to a temporary directory: the checkout may be read-only
    import __graft_entry__ as g
    if not os.path.exists(os.path.join(PKG, "libaurora_cuda.so")):
        g.build()
    exe = str(tmp_path_factory.mktemp("cpp_mirror") / "mirror_test")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "cpp", "mirror_test.cpp"),
                           "-L", PKG, "-laurora_cuda", f"-Wl,-rpath,{PKG}", "-o", exe])
    return exe


def test_cpp_mirror_builds_and_refuses_to_run_without_a_gpu(mirror_exe):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is visible here")
    r = subprocess.run([mirror_exe, os.path.join(ROOT, "tests", "golden", "Test.bmp"), "expect-no-gpu"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "aurora_init failed" in r.stdout, r.stdout + r.stderr


@pytest.mark.gpu
def test_cpp_mirror_round_trips(mirror_exe):
    r = subprocess.run([mirror_exe, os.path.join(ROOT, "tests", "golden", "Test.bmp")], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "mirror_test: 0 failures" in r.stdout, r.stdout + r.stderr
