"""-m gpu: multi-GPU evaluation of chunked tracks (SURVEY.md 8(f) rows e x f1).  Every rank sweeps the row blocks
rank (mod world) of the chunked all-vs-all sweep (the half sweep for min / max / mean, the rectangle otherwise), the
per-(query, relevant item) rank counters are summed over the ranks and finish() yields AP / R1.  Each rank runs the
same kernel on the same tiles as the single-GPU sweep, so every counter -- and so every AP / R1 -- is the same:

* ranks emulated one after the other on one GPU (counters summed by hand), half sweep and rectangle, full and ragged
  tracks, and the staged form whose relevant track similarities are computed once across the ranks;
* two PROCESSES sharing cuda:0 over gloo: evaluate_all_vs_all / evaluate_sharded through real collectives;
* real NCCL on two GPUs (skipped on a single-GPU box)."""
import os

import pytest
import torch

from oracle import evaluator as oev

pytestmark = pytest.mark.gpu


def _chunked_set(n, s, d, seed):
    from wealy_b200.data import synth
    base = synth.make_eval_set(n, d, seed=seed)
    g = torch.Generator().manual_seed(seed + 100)
    # chunk embeddings = the track embedding + chunk-level noise (some chunks of a cover match better than others)
    z = base["z"][:, None, :] + 0.8 * base["z"].norm(dim=1).mean() / d ** 0.5 * torch.randn(n, s, d, generator=g)
    return base["c"], base["i"], z.contiguous()


def _lens(n, s, seed):
    g = torch.Generator().manual_seed(seed + 500)
    return torch.randint(1, s + 1, (n,), generator=g)


# tracks per chunk count: chunk rows 3000 / 2664 / 2720, none a multiple of 256
_SIZES = {2: 1500, 8: 333, 16: 170}


def _emulated(c, i, z, world, redux, lens, staged=False):
    """Ranks 0 .. world-1 one after the other, each on a plan of its own; counters (and, staged, thresholds) summed by
    hand where a multi-GPU run all-reduces them.  -> (finish() of rank 0, the plans, the summed thresholds)."""
    from wealy_b200 import evaluation as we
    plans = [we.EvalPlan(c, i, c, i) for _ in range(world)]
    thr = None
    if staged:
        for r, pl in enumerate(plans):
            pl.shard_prepare(z, r, world, redux=redux, q_chunks=lens)
            t = pl.thresholds_tensor()
            thr = t.clone() if thr is None else thr + t
        for pl in plans:
            pl.thresholds_tensor().copy_(thr)
    total = None
    for r, pl in enumerate(plans):
        if staged:
            pl.shard_sweep(r, world)
        else:
            pl.sweep_shard(z, r, world, redux=redux, q_chunks=lens)
        cnt = pl.counts_tensor()
        assert cnt.dtype == torch.int32 and cnt.numel() == max(pl.total_pairs, 1)
        total = cnt.clone() if total is None else total + cnt
    plans[0].counts_tensor().copy_(total)
    out = plans[0].finish()
    torch.cuda.synchronize()
    return out, plans, thr


def _close(plans):
    for pl in plans:
        pl.close()


@pytest.mark.parametrize("s", [2, 8, 16])
@pytest.mark.parametrize("ragged", [False, True])
@pytest.mark.parametrize("redux", ["min", "max", "mean"])
@pytest.mark.parametrize("world", [2, 3, 8])
def test_sharded_chunked_sweep_emulated_on_one_gpu(world, redux, ragged, s):
    from wealy_b200 import evaluation as we
    n = _SIZES[s]
    c, i, z = _chunked_set(n, s, 64, seed=7 * n + s)
    lens = _lens(n, s, seed=n) if ragged else None
    cq, iq, zq = c.cuda(), i.cuda(), z.cuda()
    ref = we.EvalPlan(cq, iq, cq, iq).run(zq, zq, redux=redux, q_chunks=lens)
    out, plans, _ = _emulated(cq, iq, zq, world, redux, lens)
    assert torch.equal(out["aps"], ref["aps"]) and torch.equal(out["r1s"], ref["r1s"])
    assert torch.allclose(out["sums"], ref["sums"], rtol=1e-9)
    _close(plans)


def test_sharded_chunked_sweep_flat_layout_and_errors():
    """[N * s, D] with chunks=s is the same sweep; the sharded chunked entries refuse what the kernels do not do."""
    from wealy_b200 import evaluation as we
    n, s, d = 333, 8, 64
    c, i, z = _chunked_set(n, s, d, seed=5)
    cq, iq, zq = c.cuda(), i.cuda(), z.cuda()
    ref = we.EvalPlan(cq, iq, cq, iq).run(zq, zq, redux="max")
    plans = [we.EvalPlan(cq, iq, cq, iq) for _ in range(3)]
    for r, pl in enumerate(plans):
        pl.sweep_shard(zq.reshape(n * s, d), r, 3, redux="max", chunks=s)
    total = sum(pl.counts_tensor().clone() for pl in plans)
    plans[0].counts_tensor().copy_(total)
    out = plans[0].finish()
    assert torch.equal(out["aps"], ref["aps"]) and torch.equal(out["r1s"], ref["r1s"])
    pl = plans[0]
    with pytest.raises(NotImplementedError):
        pl.sweep_shard(zq[:, :3].contiguous(), 0, 2)                              # 3 chunks per track
    with pytest.raises(NotImplementedError):
        pl.sweep_shard(zq, 0, 2, redux="bpwr")
    with pytest.raises(AssertionError):
        we.EvalPlan(cq[:100], iq[:100], cq, iq).sweep_shard(zq, 0, 2)             # needs queries == candidates
    pl.shard_prepare(zq, 0, 4, redux="min")
    with pytest.raises(ValueError):
        pl.shard_sweep(0, 4, redux="mean")                                        # thresholds were computed for min
    torch.cuda.synchronize()
    _close(plans)


@pytest.mark.parametrize("redux", ["min", "mean", "meanmin"])
def test_sharded_chunked_rectangle_sweep(redux, monkeypatch):
    """WEALY_SYM_TRACKS=0 (and meanmin, which has no half sweep): the rectangle sweep sharded by row blocks -- every
    rank's rows complete, zeros elsewhere."""
    from wealy_b200 import evaluation as we
    monkeypatch.setenv("WEALY_SYM_TRACKS", "0")
    n, s = 333, 8
    c, i, z = _chunked_set(n, s, 64, seed=11)
    lens = _lens(n, s, seed=11)
    cq, iq, zq = c.cuda(), i.cuda(), z.cuda()
    for q_chunks in (None, lens):
        ref = we.EvalPlan(cq, iq, cq, iq).run(zq, zq, redux=redux, q_chunks=q_chunks)
        for world in (2, 3):
            out, plans, _ = _emulated(cq, iq, zq, world, redux, q_chunks)
            assert torch.equal(out["aps"], ref["aps"]) and torch.equal(out["r1s"], ref["r1s"])
            assert torch.allclose(out["sums"], ref["sums"], rtol=1e-9)
            _close(plans)


@pytest.mark.parametrize("ragged", [False, True])
@pytest.mark.parametrize("redux", ["min", "mean"])
@pytest.mark.parametrize("world", [4, 8])
def test_staged_track_thresholds(world, redux, ragged):
    """Staged form: each rank computes the relevant track similarities of its share of the queries, the shares are
    summed (by hand here), every rank rebuilds its limits / counts from the sum.  The assembled thresholds equal the
    single-GPU K_pos bit for bit; the per-item ranks (which read the counts) and AP / R1 are identical."""
    from wealy_b200 import evaluation as we
    n, s = 1500, 2
    c, i, z = _chunked_set(n, s, 64, seed=world + 3)
    lens = _lens(n, s, seed=world) if ragged else None
    cq, iq, zq = c.cuda(), i.cuda(), z.cuda()
    ref_plan = we.EvalPlan(cq, iq, cq, iq)
    ref = ref_plan.run(zq, zq, redux=redux, q_chunks=lens)
    out, plans, thr = _emulated(cq, iq, zq, world, redux, lens, staged=True)
    m = max(ref_plan.total_pairs, 1)
    assert thr.numel() == m
    assert torch.equal(thr.view(torch.int32), ref_plan.thresholds_tensor()[-m:].view(torch.int32))
    for a, b in zip(plans[0].ranks(), ref_plan.ranks()):
        assert torch.equal(a, b)
    assert torch.equal(out["aps"], ref["aps"]) and torch.equal(out["r1s"], ref["r1s"])
    assert torch.allclose(out["sums"], ref["sums"], rtol=1e-9)
    _close(plans)
    ref_plan.close()


def test_sharded_chunked_rank_bands_against_oracle():
    """One sharded case against the oracle: every R1 inside the band its 1e-5 neighbours allow, exact where the band is
    a single rank."""
    n, s, redux = 600, 4, "max"
    c, i, z = _chunked_set(n, s, 48, seed=23)
    lens = _lens(n, s, seed=23)
    out, plans, _ = _emulated(c.cuda(), i.cuda(), z.cuda(), 3, redux, lens)
    r1s = out["r1s"].cpu().double()
    lo, hi = oev.rank_tolerance(c, i, z, c, i, z, gap=1e-5, redux=redux, q_len=lens, c_len=lens)
    assert bool(((r1s >= lo) & (r1s <= hi)).all())
    exact = lo == hi
    assert int(exact.sum()) > n // 2
    aps_o, r1_o = oev.evaluate_argsort(c, i, z, c, i, z, redux=redux, q_len=lens, c_len=lens)
    assert torch.equal(r1s[exact], r1_o[exact])
    _close(plans)


def _check_ranks(wd, we, c, i, z, dev):
    """The chunked cases every multi-process test runs; -> True where every result equals the single-GPU run."""
    n, s = z.shape[0], z.shape[1]
    lens = _lens(n, s, seed=3)
    zd = z.to(dev)
    cd, id_ = c.to(dev), i.to(dev)
    ok = True
    for redux, q_chunks in (("min", None), ("meanmin", None), ("mean", lens)):
        ref = we.EvalPlan(cd, id_, cd, id_).run(zd, zd, redux=redux, q_chunks=q_chunks)
        out = wd.evaluate_all_vs_all(c, i, z.pin_memory(), redux=redux, q_chunks=q_chunks)     # pinned host input
        ok &= torch.equal(out["aps"], ref["aps"]) and torch.equal(out["r1s"], ref["r1s"]) and out["count"] == n
        if out["plan"] is not None:
            out["plan"].close()
    # top-k: the query-partitioned scheme, lists gathered
    ref = we.EvalPlan(cd, id_, cd, id_).run(zd, zd, topk=5, redux="minmean", q_chunks=lens)
    got = wd.evaluate_sharded(cd, id_, zd, cd, id_, zd, topk=5, redux="minmean", q_chunks=lens, c_chunks=lens)
    ok &= torch.equal(got["aps"], ref["aps"]) and torch.equal(got["r1s"], ref["r1s"])
    ok &= torch.equal(got["topk_idx"], ref["topk_idx"]) and float((got["topk_sim"] - ref["topk_sim"]).abs().max()) <= 2e-6
    got = wd.evaluate_all_vs_all(cd, id_, zd, topk=5, redux="min")
    ref = we.EvalPlan(cd, id_, cd, id_).run(zd, zd, topk=5, redux="min")
    ok &= torch.equal(got["aps"], ref["aps"]) and torch.equal(got["topk_idx"], ref["topk_idx"])
    # a track without a relevant candidate: every rank raises, on either route
    c_bad = cd.clone()
    c_bad[0] = 10_000_000
    for redux in ("min", "meanmin"):
        try:
            wd.evaluate_all_vs_all(c_bad, id_, zd, redux=redux)
            ok = False
        except ValueError:
            pass
    return bool(ok)


def _gloo_worker(rank, world, port, ret):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    import torch.distributed as dist
    torch.cuda.set_device(0)                                  # both ranks on the one GPU of the box
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from wealy_b200 import evaluation as we, dist as wd
        c, i, z = _chunked_set(1100, 4, 64, seed=29)
        ret[rank] = _check_ranks(wd, we, c, i, z, torch.device("cuda", 0))
        torch.cuda.synchronize()
    finally:
        dist.destroy_process_group()


def test_two_processes_one_gpu_gloo_chunked():
    import torch.multiprocessing as mp
    port = 29700 + (os.getpid() % 90)
    ret = mp.Manager().dict()
    mp.spawn(_gloo_worker, args=(2, port, ret), nprocs=2, join=True)
    assert dict(ret) == {0: True, 1: True}


def _nccl_worker(rank, world, port, ret):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        from wealy_b200 import evaluation as we, dist as wd
        c, i, z = _chunked_set(1100, 4, 64, seed=29)
        ret[rank] = _check_ranks(wd, we, c, i, z, dev)
        torch.cuda.synchronize()
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_nccl_two_ranks_chunked_match_one_gpu():
    import torch.multiprocessing as mp
    port = 29800 + (os.getpid() % 90)
    ret = mp.Manager().dict()
    mp.spawn(_nccl_worker, args=(2, port, ret), nprocs=2, join=True)
    assert dict(ret) == {0: True, 1: True}
