"""Host-side logic of multi-GPU chunked-track evaluation over a world_size-2 gloo group (no GPU): the sharded upload of
[N, s, D] tracks and the per-rank query slice of evaluate_sharded."""
import os

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from wealy_b200 import dist as wd


def _worker(rank, world, port, n, s, ret):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        z = torch.arange(n * s * 3, dtype=torch.float32).reshape(n, s, 3)
        # every rank uploads whole tracks, 1/world of them; all ranks end with the full [N, s, D] tensor
        up = wd.upload_sharded(z, torch.device("cpu"))
        ok = up.shape == (n, s, 3) and torch.equal(up, z)
        # evaluate_sharded's slice: this rank's query tracks and their chunk counts, in both layouts
        lens = torch.arange(n) % s + 1
        lo, hi = wd.shard_range(n, rank, world)
        qz, ql = wd.query_slice(z, lens, lo, hi)
        ok &= torch.equal(qz, z[lo:hi]) and torch.equal(ql, lens[lo:hi])
        qf, qlf = wd.query_slice(z.reshape(n * s, 3), lens, lo, hi, chunks=s)
        ok &= torch.equal(qf, z[lo:hi].reshape(-1, 3)) and torch.equal(qlf, lens[lo:hi])
        ok &= wd.query_slice(z, None, lo, hi)[1] is None
        # the slices of the ranks put back together are the whole set
        counts = wd.gather_rows(ql, n)
        ok &= torch.equal(counts, lens)
        ret[rank] = bool(ok)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("n,s", [(11, 4), (37, 8)])
def test_chunked_upload_and_query_slices_over_gloo_world2(n, s):
    world = 2
    port = 31500 + (os.getpid() % 2000) + n
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(world, port, n, s, ret), nprocs=world, join=True)
    assert dict(ret) == {0: True, 1: True}


def test_chunk_arguments_are_refused_before_any_collective():
    """What the kernels do not do is refused from the arguments alone -- identical on every rank."""
    with pytest.raises(NotImplementedError):
        wd._chunks_per_track(torch.zeros(10, 3, 8), None, "min", None)   # 3 chunks per track
    with pytest.raises(NotImplementedError):
        wd._chunks_per_track(torch.zeros(10, 4, 8), None, "bpwr", None)
    with pytest.raises(ValueError):
        wd._chunks_per_track(torch.zeros(10, 8), None, "min", torch.ones(10))
    with pytest.raises(ValueError):
        wd._chunks_per_track(torch.zeros(10, 4, 8), 8, "min", None)
    assert wd._chunks_per_track(torch.zeros(40, 8), 4, "meanmin", None) == 4
    assert wd._chunks_per_track(torch.zeros(10, 8), None, "min", None) == 1
