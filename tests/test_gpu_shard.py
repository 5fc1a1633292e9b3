"""SURVEY 8e behind the C ABI: hb_shard_* (native partition, schedule sort, un-permute + NCCL all-gather on a side stream).
World size 1 runs everywhere; the world-size-2 case needs two GPUs and is skipped on a single-GPU machine."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


def test_shard_world1_unpermute_and_compaction(gpu_ctx):
    import torch
    from hunter_bipedal_control_b200 import sharding
    dev = torch.device("cuda", 0)
    total = 37
    shard = sharding.Shard(gpu_ctx, None, 1, 0, total, max_row_doubles=12)
    assert (shard.lo, shard.hi) == (0, total)
    rng = np.random.default_rng(1)
    rows = rng.standard_normal((total, 10))
    perm = rng.permutation(total).astype(np.int32)
    inv = np.empty_like(perm); inv[perm] = np.arange(total, dtype=np.int32)
    d_sorted = torch.from_numpy(rows[perm]).to(dev)                  # what a schedule-sorted solve leaves behind
    d_inv = torch.from_numpy(inv).to(dev)
    for width, src in ((10, d_sorted), (12, torch.cat([d_sorted, d_sorted[:, :2]], dim=1).contiguous())):
        addr = shard.gather(src, d_inv)
        shard.wait(block_host=True)
        assert np.array_equal(shard.to_host(addr, width)[:, :10], rows)
    with pytest.raises(Exception):
        shard.gather(torch.zeros((total, 13), dtype=torch.float64, device=dev))      # wider than max_row_doubles
    shard.close()


@pytest.mark.parametrize("total", [1001])
def test_shard_world2_nccl_gather_equals_single_gpu(total):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1", "--master-port", "29617",
           os.path.join(HERE, "shard_worker.py"), str(total)]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "SHARD_OK world=2" in r.stdout
