"""Multi-GPU checks on real GPUs (NCCL): runs tests/dist_train_check.py under torchrun on every GPU of the box (>= 2).
On a one-GPU box the test is skipped; the CPU-side logic of the same code runs in tests/test_gloo_shard.py (gloo, world 2)."""
import json
import os
import socket
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_nccl_train_render_grow_identical_across_ranks():
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs in one machine")
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(n), "--master-addr", "127.0.0.1",
                        "--master-port", str(port), os.path.join(ROOT, "tests", "dist_train_check.py")], capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    line = [l for l in r.stdout.splitlines() if l.startswith("{")][-1]
    out = json.loads(line)
    assert out["world"] == n and out["render_sharded_bit_identical"] and out["grow_merge_identical"]
