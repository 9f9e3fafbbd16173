"""Data-parallel step on 2 GPUs (torchrun, NCCL) against the oracle: tests/ddp_check.py.  Skipped with fewer than 2 GPUs."""
import os
import socket
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_data_parallel_step_matches_the_oracle_on_two_gpus():
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), os.path.join(ROOT, "tests", "ddp_check.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=1500)
    print(out.stdout[-4000:])
    assert out.returncode == 0, out.stderr[-4000:]
    for mode in ("ddp", "exact", "graph"):
        assert "DDP_CHECK_OK %s" % mode in out.stdout
