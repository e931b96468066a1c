"""Host-side logic that needs no GPU: synthetic generator, query sharding and the result merge
over a world_size-2 gloo group."""
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from wealy_b200 import dist as wd
from wealy_b200.data import synth


def test_clique_multisets_match_the_shipped_splits():
    s = synth.clique_size_multiset("shs100k_test")
    assert s.sum() == 10547 and s.size == 1692 and s.min() == 2 and s.max() == 162
    s = synth.clique_size_multiset("lyric_covers_test")
    assert s.sum() == 15584 and s.size == 4913 and s.max() == 66
    assert synth.clique_size_multiset("shs100k_train").max() == 359


@pytest.mark.parametrize("n", [64, 1000, 10547, 20001])
def test_sampled_sizes_sum_and_have_no_singletons(n):
    sizes = synth.sample_clique_sizes(n, "shs100k_test", seed=3)
    assert sizes.sum() == n and sizes.min() >= 2


def test_song_id_is_the_reference_hash():
    # md5("12-3")[:4] big-endian & 0x7fffffff  (lib/embedding_dataset/utils.py:7-13)
    import hashlib
    ref = int.from_bytes(hashlib.md5(b"12-3").digest()[:4], "big") & 0x7FFFFFFF
    assert synth.deterministic_song_id(12, 3) == ref and 0 <= ref < 2 ** 31


def test_eval_set_shapes_and_determinism():
    a = synth.make_eval_set(500, 32, seed=1)
    b = synth.make_eval_set(500, 32, seed=1)
    assert a["z"].shape == (500, 32) and a["z"].dtype == torch.float32 and a["c"].dtype == torch.long
    assert torch.equal(a["z"], b["z"]) and torch.equal(a["i"], b["i"])
    counts = torch.bincount(a["c"])
    assert counts[counts > 0].min() >= 2


def test_loss_batch():
    s = synth.make_loss_batch(64, 16, seed=0, per_clique=4)
    assert s["z"].shape == (64, 16) and torch.bincount(s["label"]).max() == 4
    assert len(torch.unique(s["idx"])) == 62      # two duplicated sample ids


@pytest.mark.parametrize("n,world", [(10, 1), (10, 3), (7, 8), (500000, 8), (0, 2)])
def test_shard_range_partitions(n, world):
    spans = [wd.shard_range(n, r, world) for r in range(world)]
    assert spans[0][0] == 0 and spans[-1][1] == n
    assert all(spans[r][1] == spans[r + 1][0] for r in range(world - 1))
    lens = [hi - lo for lo, hi in spans]
    assert max(lens) - min(lens) <= 1


def _worker(rank, world, port, n, ret):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        full_ap = torch.arange(n, dtype=torch.float32) / n
        full_r1 = torch.arange(n, dtype=torch.float32) + 1
        lo, hi = wd.shard_range(n, rank, world)
        sums = torch.tensor([full_ap[lo:hi].double().sum(), full_r1[lo:hi].double().sum(), float(hi - lo)],
                            dtype=torch.float64)
        m, r1, cnt = wd.merge_sums(sums)
        aps = wd.gather_rows(full_ap[lo:hi].clone(), n)
        tk = wd.gather_rows(torch.arange(lo, hi)[:, None].repeat(1, 3), n)
        # sharded upload: every rank contributes its 1/world slice of the rows, all ranks end with the full matrix
        zfull = torch.arange(n * 5, dtype=torch.float32).reshape(n, 5)
        zup = wd.upload_sharded(zfull, torch.device("cpu"))
        # data-parallel loss: global labels in rank order, single-label noise applied to the GLOBAL batch and
        # written back into the caller's local labels in place (lib/losses.py:34-35)
        from wealy_b200.dist_losses import _gather_ids
        lab_local = torch.full((6,), 3, dtype=torch.long)
        labg, idxg = _gather_ids(lab_local, torch.arange(6) + 6 * rank, None)
        want = torch.full((12,), 3, dtype=torch.long)
        want[:2] = -1
        dp_ok = torch.equal(labg, want) and torch.equal(idxg, torch.arange(12)) and torch.equal(lab_local, want[6 * rank:6 * rank + 6])
        ok = (dp_ok and torch.equal(zup, zfull) and cnt == n and abs(m - float(full_ap.double().mean())) < 1e-12
              and abs(r1 - float(full_r1.double().mean())) < 1e-9
              and torch.equal(aps, full_ap) and torch.equal(tk[:, 0], torch.arange(n)))
        ret[rank] = bool(ok)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("n", [11, 64])
def test_merge_over_gloo_world2(n):
    world = 2
    port = 29500 + (os.getpid() % 2000)
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker, args=(world, port, n, ret), nprocs=world, join=True)
    assert dict(ret) == {0: True, 1: True}


def test_redux_string_dispatch_follows_the_reference_order():
    """lib/tensor_ops.py:291-368 tests the redux string in a fixed order ("best" swallows "bestmin", the "s" prefix comes
    last); the plan for the fused kernel must make the same choices, and leave the random / nested forms alone."""
    from wealy_b200.tensor_ops import _redux_plan
    assert _redux_plan("min") == (0, 0, 0) and _redux_plan("meanmin") == (4, 0, 0)
    assert _redux_plan("best") == (5, 1, 0) and _redux_plan("best-3") == (5, 3, 0)
    assert _redux_plan("bestmin-2") == (5, 2, 0)                  # shadowed by "best", like upstream
    assert _redux_plan("worst-2") == (6, 2, 0)
    assert _redux_plan("bpwr") == (7, 0, 0) and _redux_plan("bpwr-3") == (7, 3, 0)
    assert _redux_plan("smin") == (0, 0, 1) and _redux_plan("sbpwr-3") == (7, 3, 1) and _redux_plan("sbest-4") == (5, 4, 1)
    assert _redux_plan("randmin") is None and _redux_plan("srandmin") is None
    assert _redux_plan("ssmin") is None and _redux_plan("nope") is None and _redux_plan("s") is None


def test_bench_arms_share_one_config():
    """bench.py's GPU arm and its reference arm must describe the same workload with the same `config` dictionary."""
    import importlib.util
    ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("_bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    for n, world, tracks in ((100000, 1, 0), (282843, 8, 0), (500000, 8, 500000)):
        a, b = bench.workload_config(n, world, tracks), bench.workload_config(n, world, tracks)
        assert a == b and a["tracks"] == n and a["n_gpus"] == world and "workload" in a
    synth = bench.load_synth()
    assert hasattr(synth, "make_eval_set")


def test_bench_dump_stays_under_its_limit_with_a_fixed_sample(tmp_path, monkeypatch):
    """bench.py --dump-outputs: float32 / float64 .npy files; an output past the size limit keeps the same seeded sample
    of queries in every run, with the sampled query indices beside it."""
    import importlib.util
    ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("_bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    n = 50_000
    aps, r1s, sums = torch.rand(n), torch.arange(1, n + 1, dtype=torch.float32), torch.tensor([1.0, 2.0, 3.0], dtype=torch.float64)
    bench.dump_outputs(str(tmp_path / "full"), {"aps": aps, "r1s": r1s}, {"sums": sums})
    assert sorted(os.listdir(tmp_path / "full")) == ["aps.npy", "r1s.npy", "sums.npy"]
    assert np.load(tmp_path / "full" / "aps.npy").dtype == np.float32 and np.load(tmp_path / "full" / "sums.npy").dtype == np.float64
    assert np.array_equal(np.load(tmp_path / "full" / "aps.npy"), aps.numpy())
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 64 * 1024 + 160_000)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), {"aps": aps, "r1s": r1s}, {"sums": sums})
        assert sum(f.stat().st_size for f in (tmp_path / run).iterdir()) <= bench.DUMP_LIMIT_BYTES
    rows = np.load(tmp_path / "a" / "query_index.npy")
    assert rows.dtype == np.float64 and 0 < rows.size < n and np.all(np.diff(rows) > 0)
    for name in ("query_index", "aps", "r1s", "sums"):
        assert np.array_equal(np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy"))
    assert np.array_equal(np.load(tmp_path / "a" / "r1s.npy"), rows.astype(np.float32) + 1)
    monkeypatch.setattr("sys.argv", ["bench.py", "--steps", "0"])
    with pytest.raises(SystemExit):
        bench.main()


def test_host_route_is_only_offered_for_one_pinned_matrix(monkeypatch):
    """evaluate() hands embeddings to wealy_eval_run_host only when the device can read them itself: ONE pinned host
    matrix on both sides, big enough for the pipeline to pay; everything else keeps copy-then-compute.  (No GPU here:
    pageable tensors cover the refusals; the accepting side runs in tests/test_gpu_eval_host.py.)"""
    import torch
    from wealy_b200.evaluation import _host_streamable
    monkeypatch.setenv("WEALY_HOST_STREAM_MIN_ROWS", "8")
    c, i = torch.arange(16) // 2, torch.arange(16)
    z = torch.randn(16, 32)
    assert not _host_streamable(c, i, z, c, i, z)                       # pageable memory
    assert not _host_streamable(c, i, z, c, i, z.clone())               # two matrices
    assert not _host_streamable(c, i, z, c.clone(), i, z)               # two id sets
    assert not _host_streamable(c, i, z.numpy(), c, i, z.numpy())       # not a tensor
    assert not _host_streamable(c, i, z[:, :30], c, i, z[:, :30])       # rows of 30 elements
    monkeypatch.setenv("WEALY_HOST_STREAM", "0")
    assert not _host_streamable(c, i, z, c, i, z)
