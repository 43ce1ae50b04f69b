"""N-rank == 1-rank (NCCL all-reduce of the packed reduced system); needs >= 2 GPUs, skipped otherwise."""
import json
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("mode", ["peer", "nccl+mailbox", "nccl", "callback"])
def test_two_rank_iterations_match_single_rank_oracle(built, mode):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29533", os.path.join(ROOT, "tests", "multi_gpu_worker.py"), mode]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=150)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    line = [l for l in res.stdout.splitlines() if l.startswith("{")][-1]
    out = json.loads(line)
    assert out["ok"] and out["replicas_identical"], out
    if mode != "callback":
        assert out["comm"]["nccl"] and out["comm"]["graph"], out          # the iteration ran as a CUDA graph with NCCL inside
        assert out["comm"]["peer_mailbox"] == (mode in ("peer", "nccl+mailbox")), out
        assert out["comm"]["peer_reduce"] == (mode == "peer"), out
