"""GPU, N >= 2 (-m gpu): multi-GPU arity-4 tree build (leaf shards, NCCL all-gather per level) equals the
single-GPU build on every rank.  Skipped on boxes with one GPU (the CPU/gloo twin is tests/test_dist_cpu.py)."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _ngpu():
    import torch
    return torch.cuda.device_count()


@pytest.mark.parametrize("k", [3, 8])
def test_tree_build_dist_matches_single_gpu(k):
    n = _ngpu()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    world = 2 if n < 4 else 4
    if k == 3 and world == 4:
        world = 2
    port = 29700 + (os.getpid() % 200)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
           "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.join("tests", "dist_gpu_worker.py"), str(k)]
    res = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert "GPU_DIST_OK" in res.stdout
