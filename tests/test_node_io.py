"""The pipelined node-loop program (tests/cpp/node_loop_async.cpp) compiles against the façade and links against libmrsb.so on any
machine; without a GPU it fails loudly.  On a GPU, tests/test_node_io_gpu.py runs it."""
import os
import subprocess

import pytest

from test_cpp_facade import build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_node_loop_async_compiles_links_and_fails_loudly_without_gpu(tmp_path):
    import torch

    exe = build(tmp_path, os.path.join(ROOT, "tests", "cpp", "node_loop_async.cpp"))
    if torch.cuda.is_available():
        pytest.skip("a GPU is present: covered by the gpu test")
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 3 and "no CUDA device" in r.stderr
