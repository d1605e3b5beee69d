"""N-GPU == 1-GPU on hardware: NCCL ranks with the real kernels on shards of one corpus (needs >= 2 visible GPUs)."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_two_nccl_ranks_equal_one_gpu():
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least two GPUs")
    world = 2 if n < 4 else 4
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr",
           "127.0.0.1", "--master-port", "29533", os.path.join(ROOT, "tests", "mp_nccl_check.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert r.stdout.count("OK dropout=") == 2, r.stdout[-2000:]
