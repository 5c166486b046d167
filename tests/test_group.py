"""Multi-GPU group contexts behind the C ABI (SURVEY 8e).

CPU: the row / block maps exported by the library are plain integer functions and must agree with the host-side
partition module (which the world-size-2 gloo test in test_partition.py exercises end to end).
GPU (-m gpu): a ONE-rank group drives every code path of the in-library partitioning on a single device (block-sharded
upload -> ncclAllGather, partitioned gtp_mul -> row-sharded result -> grouped ncclBroadcast replication); with two or more
GPUs visible the same checks run under torchrun with real peers (tests/group_worker.py).
"""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_row_and_block_maps_match_the_partition_module():
    import genfer_b200
    from genfer_b200.partition import rows_for_rank, shard_bounds
    for n in (1, 7, 16, 24, 33, 300):
        for world in (1, 2, 3, 4, 8):
            seen = []
            for rank in range(world):
                rows = genfer_b200.partition_rows(n, world, rank)
                assert rows == rows_for_rank(n, world, rank)
                seen += rows
                assert genfer_b200.partition_block(n, world, rank) == shard_bounds(n, world, rank)
            assert sorted(seen) == list(range(n))


def test_folded_cyclic_rows_balance_the_macs():
    """Row k0 costs k0 + 1 sub-products (:1001-1010): with 2W | rows every rank gets the same total."""
    import genfer_b200
    for n, world in ((16, 2), (16, 4), (16, 8), (24, 4), (32, 8)):
        loads = [sum(k + 1 for k in genfer_b200.partition_rows(n, world, r)) for r in range(world)]
        assert len(set(loads)) == 1, (n, world, loads)


@pytest.mark.gpu
def test_one_rank_group_drives_the_partitioned_paths():
    import genfer_b200
    from oracle import oracle as O
    from helpers import synth_uniform
    uid = genfer_b200.nccl_unique_id()
    ctx = genfer_b200.Context.create_group(0, 0, 1, uid)
    try:
        assert ctx.group_info()[:2] == (0, 1)
        ctx.set_partition_threshold(0)
        shape = (8, 6, 16, 16)
        x, y = synth_uniform(shape, 5), synth_uniform(shape, 6)
        X = genfer_b200.TaylorPoly.from_host_block_ptr(x.ctypes.data, shape, shape, ctx)
        Y = genfer_b200.TaylorPoly.new(y, shape, ctx)
        assert X.is_distributed()
        Z = X * Y
        assert Z.is_distributed() and not X.is_distributed()
        assert Z.local_rows() == list(range(8))
        ref = (O.taylor(x) * O.taylor(y)).array()
        local = np.empty(shape)
        Z.to_host_local_ptr(local.ctypes.data)
        np.testing.assert_allclose(local, ref, rtol=1e-12)
        W = Z * Y                                   # Horner-style chain: Z is replicated here, W is sharded again
        assert W.is_distributed() and not Z.is_distributed()
        np.testing.assert_allclose(W.array(), (O.taylor(ref) * O.taylor(y)).array(), rtol=1e-12)
        _, _, products, gathers = ctx.group_info()
        assert products == 2 and gathers >= 3
    finally:
        ctx.close()


@pytest.mark.gpu
def test_two_rank_group_under_torchrun():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29611", os.path.join(ROOT, "tests", "group_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "group worker ok" in r.stdout
