"""Multi-GPU parity (needs >= 2 B200s on the machine: NCCL does not put two ranks on one device; on a single-GPU machine the test
is skipped by tests/conftest.py and tests/test_gpu_exchange.py covers the same exchange with ranks sharing cuda:0): launches
tools/shard_check.py with one process per GPU over NCCL."""
import os
import subprocess
import sys

import pytest

pytestmark = [pytest.mark.gpu, pytest.mark.multigpu]
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_two_gpu_sharded_search_matches_oracle():
    import torch
    n = torch.cuda.device_count()
    assert n >= 2, "multigpu tests are skipped on machines with one GPU (tests/conftest.py)"
    world = 2 if n < 4 else 4
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", "29631", os.path.join(ROOT, "tools", "shard_check.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0 and "shard_check OK" in res.stdout, res.stdout[-2000:] + res.stderr[-2000:]
