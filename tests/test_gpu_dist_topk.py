"""-m gpu: multi-GPU all-vs-all top-k on the row-block-sharded symmetric sweep.  Every rank sweeps the row blocks
rank (mod world) with the top-k epilogue (the sampled per-query bounds are computed identically on every rank), the
rank counters are summed, and each query's local lists of all ranks are merged (topk_merge_kernel).  Every tile is
computed once, by the same kernel as on one GPU, so AP / R1 and the top-k similarities are bit-identical to the
single-GPU symmetric top-k sweep, and the indices agree wherever similarities are not exactly tied:

* ranks emulated one after the other on one GPU (counters summed, lists merged by hand), against the single-GPU run and
  the oracle;
* the merge kernel on synthetic lists: order of the lists, ties, short and overflowed lists;
* what is not eligible is refused before any work;
* two PROCESSES sharing cuda:0 over gloo, and real NCCL on two GPUs (skipped on a single-GPU box): evaluate_all_vs_all
  on the new route and on its fallback."""
import os

import pytest
import torch

from oracle import evaluator as oev

pytestmark = pytest.mark.gpu


def _set(n, d, seed, **kw):
    from wealy_b200.data import synth
    return synth.make_eval_set(n, d, seed=seed, device="cuda", **kw)


def _emulated(c, i, z, world, k):
    """Ranks 0 .. world-1 one after the other, each on a plan of its own; counters summed and lists merged by hand where
    a multi-GPU run all-reduces / exchanges them.  -> (finish() with topk_idx / topk_sim, failed queries, local lists)."""
    from wealy_b200 import evaluation as we
    plan0 = we.EvalPlan(c, i, c, i)
    total, locs = None, []
    for r in range(world):
        pl = plan0 if r == 0 else we.EvalPlan(c, i, c, i)
        loc = pl.sweep_shard_topk(z, r, world, k)
        assert pl.last_topk_path() == 1
        st = pl.stage_ms()
        assert st["topk_finalize"] > 0 and st["ap_reduce"] >= 0
        locs.append(loc)
        cnt = pl.counts_tensor()
        total = cnt.clone() if total is None else total + cnt
        if r:
            torch.cuda.synchronize()
            pl.close()
    plan0.counts_tensor().copy_(total)
    out = plan0.finish()
    idx, sim, failed = we.merge_topk(torch.stack([l["val"] for l in locs]), torch.stack([l["idx"] for l in locs]),
                                     torch.stack([l["cnt"] for l in locs]))
    out["topk_idx"], out["topk_sim"] = idx, sim
    torch.cuda.synchronize()
    plan0.close()
    return out, failed, locs


def _untied(sim):
    """Positions whose similarity differs from both neighbours in the row; the last position also depends on the
    (k + 1)-th best, which no list shows."""
    ok = torch.ones_like(sim, dtype=torch.bool)
    ok[:, 1:] &= sim[:, 1:] != sim[:, :-1]
    ok[:, :-1] &= sim[:, :-1] != sim[:, 1:]
    ok[:, -1] = False
    return ok


def _same_as_single(got, ref):
    ok = torch.equal(got["aps"], ref["aps"]) and torch.equal(got["r1s"], ref["r1s"])
    ok &= torch.equal(got["topk_sim"], ref["topk_sim"])
    m = _untied(ref["topk_sim"])
    ok &= torch.equal(got["topk_idx"][m], ref["topk_idx"][m])
    return bool(ok)


@pytest.mark.parametrize("world", [2, 3, 8])
@pytest.mark.parametrize("n,d,k", [(20000, 96, 10), (33000, 64, 128)])
def test_sharded_topk_emulated_on_one_gpu(n, d, k, world):
    from wealy_b200 import evaluation as we
    if world * k > 1024:
        pytest.skip("world * k > 1024 is not eligible (tested below)")
    s = _set(n, d, seed=60 + k)
    c, i, z = s["c"], s["i"], s["z"]
    plan = we.EvalPlan(c, i, c, i)
    ref = plan.run(z, z, topk=k)
    assert plan.last_topk_path() == 1
    torch.cuda.synchronize()
    plan.close()
    out, failed, locs = _emulated(c, i, z, world, k)
    assert failed == 0
    # every rank holds a part of the lists; together exactly the single-GPU candidates
    cnt = torch.stack([l["cnt"] for l in locs])
    assert bool((cnt >= 0).all()) and bool((cnt.sum(0) >= k).all())
    assert _same_as_single(out, ref)
    assert torch.allclose(out["sums"], ref["sums"], rtol=1e-9)
    # a query sample against the oracle: similarities within 4e-6, indices exact where neighbours are 1e-5 apart
    qs = torch.randperm(n, generator=torch.Generator().manual_seed(world))[:64]
    cc, ic, zc = c.cpu(), i.cpu(), z.cpu()
    _, _, idx_o, sim_o = oev.evaluate_argsort(cc[qs], ic[qs], zc[qs], cc, ic, zc, topk=k)
    idx, sim = out["topk_idx"].cpu()[qs], out["topk_sim"].cpu()[qs]
    assert (sim - sim_o).abs().max() <= 4e-6
    gap = torch.ones_like(idx_o, dtype=torch.bool)
    gap[:, 1:] &= (sim_o[:, :-1] - sim_o[:, 1:]) > 1e-5
    gap[:, :-1] &= (sim_o[:, :-1] - sim_o[:, 1:]) > 1e-5
    gap[:, -1] = False
    assert float(gap.float().mean()) > 0.5
    assert torch.equal(idx[gap], idx_o[gap])
    assert bool((idx != qs[:, None]).all())


def _merge_ref(val, idx, k):
    """Reference merge on the host: per query, the k best of all lists by (descending similarity, ascending index)."""
    w, n, kk = val.shape
    v = val.permute(1, 0, 2).reshape(n, w * kk).double()
    x = idx.permute(1, 0, 2).reshape(n, w * kk).long()
    order = torch.argsort(x, dim=1, stable=True)                 # secondary key first ...
    v, x = v.gather(1, order), x.gather(1, order)
    order = torch.argsort(-v, dim=1, stable=True)                # ... then the primary, stably
    return x.gather(1, order)[:, :k], v.gather(1, order)[:, :k].float()


def test_merge_kernel_on_synthetic_lists():
    from wealy_b200 import evaluation as we
    g = torch.Generator().manual_seed(3)
    for world, n, k in ((3, 200, 8), (8, 100, 128), (2, 300, 1), (5, 64, 37)):
        # few distinct similarities: ties everywhere, inside the lists, across lists and at the k-th place
        val = (torch.randint(0, 12, (world, n, k), generator=g).float() / 12.0)
        idx = torch.stack([torch.randperm(100_000, generator=g)[: world * k] for _ in range(n)]).view(n, world, k)
        idx = idx.permute(1, 0, 2).int().contiguous()
        cnt = torch.full((world, n), k, dtype=torch.int32)
        ref_idx, ref_sim = _merge_ref(val, idx, k)
        got_idx, got_sim, failed = we.merge_topk(val.cuda(), idx.cuda(), cnt.cuda())
        assert failed == 0
        assert torch.equal(got_idx.cpu(), ref_idx) and torch.equal(got_sim.cpu(), ref_sim)
        perm = torch.randperm(world, generator=g)
        p_idx, p_sim, _ = we.merge_topk(val[perm].cuda(), idx[perm].cuda(), cnt[perm].cuda())
        assert torch.equal(p_idx, got_idx) and torch.equal(p_sim, got_sim)
    # an exact tie at the k-th place goes to the lower index, whichever list holds it
    val = torch.tensor([[[0.9, 0.5]], [[0.5, 0.1]]])
    two = torch.full((2, 1), 2, dtype=torch.int32).cuda()
    for idx in (torch.tensor([[[4, 9]], [[2, 3]]]), torch.tensor([[[4, 2]], [[9, 3]]])):
        got_idx, got_sim, failed = we.merge_topk(val.cuda(), idx.int().cuda(), two)
        assert failed == 0 and got_idx.cpu().tolist() == [[4, 2]]
        assert torch.equal(got_sim.cpu(), torch.tensor([[0.9, 0.5]]))
    # ... and a run of equal similarities is ordered by index
    val = torch.tensor([[[0.9, 0.5, 0.5]], [[0.5, 0.1, 0.0]]])
    idx = torch.tensor([[[4, 9, 7]], [[8, 3, 1]]]).int()
    got_idx, got_sim, _ = we.merge_topk(val.cuda(), idx.cuda(), torch.full((2, 1), 3, dtype=torch.int32).cuda())
    assert got_idx.cpu().tolist() == [[4, 7, 8]] and torch.equal(got_sim.cpu(), torch.tensor([[0.9, 0.5, 0.5]]))


def test_merge_kernel_reports_short_and_overflowed_lists():
    from wealy_b200 import evaluation as we
    world, n, k = 3, 5, 4
    ninf = float("-inf")
    val = torch.full((world, n, k), ninf)
    idx = torch.full((world, n, k), -1, dtype=torch.int32)
    cnt = torch.zeros((world, n), dtype=torch.int32)
    for q in range(n):
        for w in range(world):
            m = [(2, 1, 1), (1, 1, 1), (4, 0, 0), (2, 1, 1), (1, 0, 0)][q][w]   # counts summing to 4, 3, 4, 4, 1
            val[w, q, :m] = torch.linspace(0.9, 0.1, m) - 0.01 * w
            idx[w, q, :m] = torch.arange(m, dtype=torch.int32) + 10 * w
            cnt[w, q] = m
    cnt[1, 3] = -1                                                # an overflowed list
    got_idx, got_sim, failed = we.merge_topk(val.cuda(), idx.cuda(), cnt.cuda())
    assert failed == 3                                            # queries 1 and 4 short, query 3 overflowed
    assert got_idx.cpu()[4].tolist() == [0, -1, -1, -1] and got_sim.cpu()[4, 1:].tolist() == [ninf] * 3
    assert got_idx.cpu()[2].tolist() == [0, 1, 2, 3]
    with pytest.raises(NotImplementedError):                     # world * k > 1024
        we.merge_topk(torch.zeros(9, 2, 128).cuda(), torch.zeros(9, 2, 128, dtype=torch.int32).cuda(),
                      torch.zeros(9, 2, dtype=torch.int32).cuda())


def _dup_set():
    """18 000 tracks, the first 3 000 exact duplicates of one another: their lists overflow."""
    s = _set(18000, 64, seed=71, md5_ids=False)
    z = s["z"].clone()
    z[:3000] = z[0]
    return s["c"], s["i"], z


def test_sharded_topk_overflow_is_reported():
    c, i, z = _dup_set()
    out, failed, locs = _emulated(c, i, z, 2, 20)
    cnt = torch.stack([l["cnt"] for l in locs])
    bad = (cnt == -1).any(0) | (cnt.clamp(min=0).sum(0) < 20)     # overflowed on some rank, or short together
    assert failed > 0 and failed == int(bad.sum())
    assert bool(bad[:3000].any())                                   # the duplicates (and some of their neighbours)


def test_ineligible_calls_are_refused():
    from wealy_b200 import evaluation as we
    s = _set(33000, 64, seed=5)
    c, i, z = s["c"], s["i"], s["z"]
    plan = we.EvalPlan(c, i, c, i)
    with pytest.raises(NotImplementedError):
        plan.sweep_shard_topk(z, 0, 9, 128)                       # world * k > 1024
    with pytest.raises(NotImplementedError):
        plan.sweep_shard_topk(z, 0, 2, 129)                       # k > 128
    os.environ["WEALY_SYM_TOPK"] = "0"
    try:
        with pytest.raises(NotImplementedError):
            plan.sweep_shard_topk(z, 0, 2, 10)
    finally:
        del os.environ["WEALY_SYM_TOPK"]
    plan.close()
    small = _set(3000, 64, seed=6)
    plan = we.EvalPlan(small["c"], small["i"], small["c"], small["i"])
    with pytest.raises(NotImplementedError):
        plan.sweep_shard_topk(small["z"], 0, 2, 10)               # N below the size threshold
    plan.close()


def _check_routes(wd, we, dev):
    """The cases every multi-process test runs; -> True where every result is what it should be."""
    ok = True
    s = _set(20000, 96, seed=61)
    c, i, z = s["c"].to(dev), s["i"].to(dev), s["z"].to(dev)
    plan = we.EvalPlan(c, i, c, i)
    ref = plan.run(z, z, topk=10)
    ok &= plan.last_topk_path() == 1
    plan.close()
    got = wd.evaluate_all_vs_all(c.cpu(), i.cpu(), z.cpu().pin_memory(), topk=10)          # pinned host input
    ok &= got["topk_path"] == "sym_sharded" and got["count"] == 20000
    ok &= _same_as_single(got, ref)
    got["plan"].close()
    # overflowing lists: every rank falls back to the query-partitioned scheme
    c, i, z = (t.to(dev) for t in _dup_set())
    got = wd.evaluate_all_vs_all(c, i, z, topk=20)
    ref = wd.evaluate_sharded(c, i, z, c, i, z, topk=20)
    ok &= got["topk_path"] == "query_sharded_fallback"
    ok &= torch.equal(got["aps"], ref["aps"]) and torch.equal(got["r1s"], ref["r1s"])
    ok &= torch.equal(got["topk_idx"], ref["topk_idx"]) and torch.equal(got["topk_sim"], ref["topk_sim"])
    # below the size threshold: today's route
    got = wd.evaluate_all_vs_all(c[:3000], i[:3000], z[:3000], topk=5, allow_empty=True)
    ok &= got["topk_path"] == "query_sharded"
    return bool(ok)


def _gloo_worker(rank, world, port, ret):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    import torch.distributed as dist
    torch.cuda.set_device(0)                                  # both ranks on the one GPU of the box
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from wealy_b200 import evaluation as we, dist as wd
        ret[rank] = _check_routes(wd, we, torch.device("cuda", 0))
        torch.cuda.synchronize()
    finally:
        dist.destroy_process_group()


def test_two_processes_one_gpu_gloo_topk():
    import torch.multiprocessing as mp
    port = 29600 + (os.getpid() % 90)
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
        ret[rank] = _check_routes(wd, we, dev)
        torch.cuda.synchronize()
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_nccl_two_ranks_topk_match_one_gpu():
    import torch.multiprocessing as mp
    port = 29900 + (os.getpid() % 90)
    ret = mp.Manager().dict()
    mp.spawn(_nccl_worker, args=(2, port, ret), nprocs=2, join=True)
    assert dict(ret) == {0: True, 1: True}
