"""The C++ host mirror (include/demi_b200.hpp) compiles against the C ABI and behaves like the reference classes."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "tests", "cpp", "host_mirror_test")


def build(native):
    native.lib()
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I" + os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "host_mirror_test.cpp"), "-o", EXE,
                           "-L" + os.path.join(ROOT, "demi_b200"), "-ldemi_b200",
                           "-Wl,-rpath," + os.path.join(ROOT, "demi_b200")])


def test_cpp_mirror_builds_and_refuses_to_run_without_a_gpu(native):
    build(native)
    if native.lib().demi_device_count() > 0:
        pytest.skip("a CUDA device is present (covered by the gpu test)")
    out = subprocess.run([EXE], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0 and "no-fallback contract" in out.stdout, out.stdout + out.stderr


@pytest.mark.gpu
def test_cpp_mirror_pipeline_on_gpu(native, tmp_path):
    build(native)           # always: a binary left by an earlier run may predate the header
    out = subprocess.run([EXE, str(tmp_path / "experiment")], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and out.stdout.strip().endswith("OK"), out.stdout + out.stderr
