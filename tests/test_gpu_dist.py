"""Multi-GPU (NCCL) parity of the sharded paths; needs >= 2 visible GPUs and skips on a one-GPU machine."""
import os
import socket
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.mark.timeout(600)
def test_sharded_paths_nccl():
    n_gpu = torch.cuda.device_count()
    if n_gpu < 2:
        pytest.skip("needs >= 2 GPUs")
    world = 4 if n_gpu >= 4 else 2
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.join(HERE, "_nccl_worker.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=580)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    for r in range(world):
        assert f"rank {r} ok" in res.stdout
