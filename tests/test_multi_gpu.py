"""SURVEY §8e equality target on real GPUs: R ranks x B patches == one process on the concatenated R*B batch
(d_losses, g_loss, post-PCGrad / task-specific / generator gradients), NCCL over NVLink, every visible GPU (up to 8).
Skipped on boxes with one GPU; the host-side choreography is covered on CPU by tests/test_distributed_gloo.py."""
import os
import socket
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_ranks_equal_single_process_on_concatenated_batch():
    n = min(8, torch.cuda.device_count())
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}", "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), os.path.join(ROOT, "tools", "check_multi_gpu.py")]
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=900)
    print(r.stdout[-4000:])
    print(r.stderr[-2000:], file=sys.stderr)
    assert r.returncode == 0 and "MULTI_GPU_CHECK PASS" in r.stdout
