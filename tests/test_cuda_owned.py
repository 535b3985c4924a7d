"""The chain engine's owner types (iq_tool_b200/csrc/cuda_owned.hpp) keep no capacity without memory behind it: a grow()
that fails returns the CUDA error and leaves the array empty, so the call that reported the error can be retried without
a fault, a leak or a double free.  Host program compiled for sm_100a; runs with or without a GPU."""
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_failed_grow_leaves_the_array_empty(tmp_path):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    exe = tmp_path / "cuda_owned_check"
    subprocess.run([nvcc, "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-I", os.path.join(ROOT, "iq_tool_b200", "csrc"),
                    "-o", str(exe), os.path.join(ROOT, "tests", "native", "cuda_owned_check.cu")], check=True,
                   stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    out = subprocess.run([str(exe)], capture_output=True, text=True)
    assert out.returncode == 0 and out.stdout.strip().endswith("OK"), out.stdout
