"""Snapshots without a GPU: the C++ branching loop through the façade compiles, links and fails loudly; the GPU side is
tests/test_snapshot_gpu.py."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_snapshot_loop_compiles_links_and_fails_loudly_without_gpu(tmp_path):
    import torch
    from test_cpp_facade import build

    exe = build(tmp_path, os.path.join(ROOT, "tests", "cpp", "snapshot_loop.cpp"))
    if torch.cuda.is_available():
        pytest.skip("a GPU is present: covered by the gpu test")
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 3 and "no CUDA device" in r.stderr
