"""CPU, gloo: unet.syncbn decides like torch.nn.SyncBatchNorm when to synchronise, and sums statistics tables of
different row counts (ranks with unequal shards) with the pixel counts of every rank."""
import os

import torch
import torch.distributed as dist
import torch.multiprocessing as mp
import torch.nn as nn


def test_no_process_group_means_per_rank_statistics():
    from unet import syncbn
    bn = nn.SyncBatchNorm(8)
    assert not dist.is_initialized()
    assert syncbn.group_of(bn.train()) is None
    assert syncbn.group_of(nn.BatchNorm2d(8).train()) is None


def _worker(rank, world, root):
    dist.init_process_group("gloo", init_method=f"file://{root}/init", rank=rank, world_size=world)
    try:
        from unet import syncbn
        bn = nn.SyncBatchNorm(4)
        assert syncbn.group_of(bn.train()) is dist.group.WORLD
        assert syncbn.group_of(bn.eval()) is None                        # eval: running statistics, no sync
        single = dist.new_group([0])
        bn1 = nn.SyncBatchNorm(4, process_group=single).train()
        if rank == 0:
            assert syncbn.group_of(bn1) is None                          # a group of one rank
        assert syncbn.group_of(nn.BatchNorm2d(4).train()) is None
        rows = (3, 5)[rank]
        table = torch.arange(rows * 2 * 4, dtype=torch.float64).reshape(rows, 2, 4) + 1000 * rank
        out, count = syncbn.exchange(table.clone(), (30, 10)[rank], dist.group.WORLD)
        torch.save({"out": out, "count": count}, f"{root}/r{rank}.pt")
    finally:
        dist.destroy_process_group()


def test_unequal_tables_are_padded_and_summed(tmp_path):
    mp.spawn(_worker, args=(2, str(tmp_path)), nprocs=2, join=True)
    r0, r1 = (torch.load(tmp_path / f"r{r}.pt", weights_only=False) for r in range(2))
    t0 = torch.arange(3 * 2 * 4, dtype=torch.float64).reshape(3, 2, 4)
    t1 = torch.arange(5 * 2 * 4, dtype=torch.float64).reshape(5, 2, 4) + 1000
    want = t1.clone()
    want[:3] += t0
    for r in (r0, r1):
        assert r["count"] == 40
        assert torch.equal(r["out"], want)
        # the column sums the finalize kernels fold are those of the two tables together
        assert torch.equal(r["out"].sum(0), t0.sum(0) + t1.sum(0))
