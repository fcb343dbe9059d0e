"""The C++ host side above the C ABI (include/b200ba_shim.hpp) compiles, links and behaves."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _build_example(tmp_path):
    from camera_calibration_b200 import build
    build.build()
    exe = str(tmp_path / "b200ba_shim_example")
    lib_dir = os.path.join(ROOT, "camera_calibration_b200", "csrc")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "shim_example.cc"), "-o", exe, "-L", lib_dir, "-lb200ba",
                           f"-Wl,-rpath,{lib_dir}"])
    return exe


def test_shim_compiles_and_fails_loudly_without_gpu(tmp_path):
    import torch
    exe = _build_example(tmp_path)
    r = subprocess.run([exe], capture_output=True, text=True)
    if torch.cuda.is_available():
        assert r.returncode == 0, r.stdout + r.stderr
    else:
        assert r.returncode == 3 and "no CUDA device" in r.stdout


@pytest.mark.gpu
def test_shim_optimize_jointly_gpu(tmp_path):
    exe = _build_example(tmp_path)
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "cost after" in r.stdout
