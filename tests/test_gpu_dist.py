"""Multi-GPU parity (needs >= 2 GPUs; skips on a machine with one): the dst-partitioned NCCL path
equals the single-GPU path on the same graph (tools/check_dist_gpu.py)."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.timeout(600)
def test_two_rank_nccl_matches_single_gpu():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29533",
                        os.path.join(ROOT, "tools", "check_dist_gpu.py")], capture_output=True, text=True, timeout=550)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "dist parity ok" in r.stdout
