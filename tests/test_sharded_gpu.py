"""GPU (>= 2 devices): row-sharded embeddings over NCCL all-to-all + data-parallel dense part against
the CPU oracle on the global batch (tests/dist_check.py under torchrun)."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("mode", ["peer", "a2a"])     # NVLink peer mappings (default) / NCCL all-to-all
def test_sharded_deepfm_matches_global_batch_oracle(cuda, mode):
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    world = 2 if n < 4 else 4
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
           "--master-addr", "127.0.0.1", "--master-port", "29631", os.path.join(ROOT, "tests", "dist_check.py")]
    env = dict(os.environ, B2CTR_SHARD_MODE=mode)
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "dist_check OK" in r.stdout and ("mode %s" % mode) in r.stdout
