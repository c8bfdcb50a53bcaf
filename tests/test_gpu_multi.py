"""Item-sharded multi-GPU parity (SURVEY 8(d) gate iv): launches tests/multi_gpu_check.py under torchrun on two
devices when the box has them (the CPU-side coverage of the same exchanges is tests/test_dist_gloo.py)."""
import os
import socket
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def test_two_gpu_sharded_parity():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", str(_free_port()), os.path.join(ROOT, "tests", "multi_gpu_check.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    sys.stdout.write(out.stdout[-4000:])
    sys.stderr.write(out.stderr[-4000:])
    assert out.returncode == 0 and "MULTI_GPU_OK" in out.stdout
