"""GPU (NCCL, world size 2) test of the gradient all-reduce (ADVICE r1): runs scripts/check_allreduce_nccl.py under
torchrun on a machine with two GPUs; skipped with fewer."""
import os
import socket
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_gradient_allreduce_nccl_world2():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "scripts", "check_allreduce_nccl.py")],
                       capture_output=True, text=True, timeout=600)
    print(r.stdout[-2000:], r.stderr[-2000:])
    assert r.returncode == 0 and "-> ok" in r.stdout
