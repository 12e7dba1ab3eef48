"""The C ABI driven by a compiled host (tests/c_host/abi_known_answers.c, plain C against include/bourse_b200.h): what a
Rust `extern "C"` binding of the reference would call, with no Python between the host and the library.  The CPU test
builds it and checks that it fails loudly without a GPU; the GPU test runs its known-answer checks."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "c_host", "abi_known_answers.c")


def _build(out_dir) -> str:
    """Compile the host into `out_dir` (the repository tree may be read-only) and return the executable's path."""
    from bourse_b200 import build

    build.build_lib()
    libdir = os.path.join(ROOT, "bourse_b200")
    exe = os.path.join(str(out_dir), "abi_known_answers")
    cmd = ["gcc", "-O1", "-Wall", "-Wextra", "-std=c11", "-I", os.path.join(ROOT, "include"), SRC, "-o", exe,
           "-L", libdir, "-lbourse_b200", f"-Wl,-rpath,{libdir}"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    assert "warning" not in res.stderr, res.stderr
    return exe


def test_c_host_builds_and_refuses_to_run_without_a_gpu(tmp_path):
    import torch

    exe = _build(tmp_path)
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    res = subprocess.run([exe], capture_output=True, text=True)
    assert res.returncode == 3 and "no CPU fallback" in res.stderr, (res.returncode, res.stderr)


@pytest.mark.gpu
def test_c_host_known_answers(tmp_path):
    exe = _build(tmp_path)
    res = subprocess.run([exe], capture_output=True, text=True)
    assert res.returncode == 0, res.stdout + res.stderr
    assert res.stdout.split() == ["ok", "order_book_trades", "ok", "env", "ok", "numpy_arrays"]


@pytest.mark.gpu
def test_c_host_multi_gpu_gather(tmp_path):
    """Multi-GPU behind the C ABI, torch-free: shards on separate devices (two when the box has them, else one), in-kernel
    agents keyed by global env id, statistics all-gathered by bb_gather_stats (ncclAllGather inside the library)."""
    import ctypes

    exe = _build(tmp_path)
    n = ctypes.c_int(0)
    assert ctypes.CDLL("libcuda.so.1").cuInit(0) == 0 and ctypes.CDLL("libcuda.so.1").cuDeviceGetCount(ctypes.byref(n)) == 0
    res = subprocess.run([exe, "--multi-gpu", str(n.value)], capture_output=True, text=True)
    assert res.returncode == 0, res.stdout + res.stderr
    assert res.stdout.split()[-2:] == ["ok", f"multi_gpu_gather_{min(n.value, 2)}_shards"]   # (NCCL prints its version banner first)
