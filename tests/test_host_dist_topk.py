"""Host-side logic of the multi-GPU all-vs-all top-k over a gloo group (no GPU): exchange_topk hands rank r the lists
of every rank for its query slice shard_range(n, r, world), list w from rank w, for even and uneven splits."""
import os

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from wealy_b200 import dist as wd


def _local_lists(rank, n, k):
    """What rank `rank` would hold after its sweep: values that name (rank, row, column)."""
    rows = torch.arange(n)[:, None].float()
    cols = torch.arange(k)[None, :].float()
    val = rank * 1000.0 + rows + cols / 128.0
    idx = (rank * 100_000 + torch.arange(n)[:, None] * 100 + torch.arange(k)[None, :]).int()
    cnt = (rank * 1000 + torch.arange(n)).int()
    return val, idx, cnt


def _worker(rank, world, port, n, k, ret):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        val, idx, cnt = _local_lists(rank, n, k)
        got_val, got_idx, got_cnt = wd.exchange_topk(val, idx, cnt)
        lo, hi = wd.shard_range(n, rank, world)
        ok = got_val.shape == (world, hi - lo, k) and got_idx.shape == (world, hi - lo, k)
        ok &= got_cnt.shape == (world, hi - lo)
        ok &= got_val.dtype == torch.float32 and got_idx.dtype == torch.int32 and got_cnt.dtype == torch.int32
        for w in range(world):
            v, i, c = _local_lists(w, n, k)
            ok &= torch.equal(got_val[w], v[lo:hi]) and torch.equal(got_idx[w], i[lo:hi]) and torch.equal(got_cnt[w], c[lo:hi])
        ret[rank] = bool(ok)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world,n,k", [(2, 11, 3), (2, 1, 4), (2, 64, 128), (3, 10, 5)])
def test_topk_list_exchange_slices_over_gloo(world, n, k):
    port = 32500 + (os.getpid() % 2000) + 7 * n + k + world
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(world, port, n, k, ret), nprocs=world, join=True)
    assert dict(ret) == {r: True for r in range(world)}
