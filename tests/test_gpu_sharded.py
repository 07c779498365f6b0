"""Multi-GPU: a pool sharded over 2 GPUs (one process per GPU, NVLink P2P mailboxes, device
barrier per tick) must end in exactly the state of the same pool on one GPU (SURVEY §8e)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_sharded_equals_single_gpu():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    world = 2
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", "29517",
           os.path.join(ROOT, "tests", "sharded_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=1200, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    line = [l for l in r.stdout.splitlines() if l.startswith("{")][-1]
    res = json.loads(line)
    assert res["ok"] and res["world"] == world
