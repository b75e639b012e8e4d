"""-m gpu, needs >= 2 GPUs on the box (skipped otherwise): the ancestral DDPM loop (`p_sample_loop`) on one clip frame-sharded over
2 ranks (torchrun, one rank per GPU, NCCL), eager and as replayed graph segments, against the single-GPU loop with the same
noise.  The checks live in tools/shard_ddpm_test.py (they assert on rank 0)."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_two_rank_ddpm_loop_matches_single_gpu():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29614", os.path.join(ROOT, "tools", "shard_ddpm_test.py")]
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=900)
    print(r.stdout[-3000:])
    assert r.returncode == 0, r.stderr[-3000:]
    assert "[ddpm]" in r.stdout
