"""-m gpu: chunked tracks with 32 chunks per track (SURVEY.md 8(f) row f1) on every evaluation path.  At s = 32 one
epilogue warp's 32 rows are exactly one query track and one 32-column chunk exactly one candidate track, and K_pos
contracts every relevant pair as 2 x 4 m16n8k16 tiles.  Checked against the oracle evaluator fed with the restated
distance_tensor_redux (lib/tensor_ops.py:288-373), against the s = 16 path on the same data, and across the half sweep /
rectangle, multi-GPU (ranks emulated on one device) and pipeline entries."""
import pytest
import torch

from oracle import evaluator as oev

pytestmark = pytest.mark.gpu

S = 32
REDUX = ["min", "max", "mean", "meanmin", "minmean"]
HALF = ["min", "max", "mean"]                    # d(q, c) == d(c, q): the all-vs-all half sweep


def _chunked_set(n, s, d, seed):
    from wealy_b200.data import synth
    base = synth.make_eval_set(n, d, seed=seed)
    g = torch.Generator().manual_seed(seed + 100)
    # chunk embeddings = the track embedding + chunk-level noise (some chunks of a cover match better than others)
    z = base["z"][:, None, :] + 0.8 * base["z"].norm(dim=1).mean() / d ** 0.5 * torch.randn(n, s, d, generator=g)
    return base["c"], base["i"], z.contiguous()


def _pad_with_junk(z, lens, c, seed):
    """Overwrite the padding chunks (index >= lens[t]) of every track: large random rows for even tracks, for odd ones
    a copy of a chunk of a track of ANOTHER clique (a near-perfect match that would move min / max if it were used)."""
    g = torch.Generator().manual_seed(seed)
    n, s, d = z.shape
    z = z.clone()
    for t in range(n):
        k = s - int(lens[t])
        if k == 0:
            continue
        if t % 2 == 0:
            z[t, int(lens[t]):] = 1e3 * torch.randn(k, d, generator=g)
        else:
            other = int(torch.nonzero(c != c[t])[0])
            z[t, int(lens[t]):] = z[other, 0]
    return z.contiguous()


def _lens_spanning(n, seed):
    """1 .. 32 valid chunks, with 1, 16, 17 and 32 each present several times."""
    g = torch.Generator().manual_seed(seed)
    lens = torch.randint(1, S + 1, (n,), generator=g)
    for k, v in enumerate((1, 16, 17, 32) * 3):
        lens[7 * k + 3] = v
    return lens


def _check_r1(r1s, c, i, z, redux, lens=None):
    lo, hi = oev.rank_tolerance(c, i, z, c, i, z, gap=1e-5, redux=redux, q_len=lens, c_len=lens)
    assert bool(((r1s >= lo) & (r1s <= hi)).all())
    exact = lo == hi
    return exact, lo


def _check_all_item_ranks(plan, c, i, z, redux, lens=None):
    """Every relevant item's rank (plan.ranks() of the last run) inside the band its 1e-5 neighbours allow, exact where
    the band is a single rank; its threshold within 4e-6 of the oracle's reduced similarity."""
    off_g, ranks_g, sims_g = (t.cpu() for t in plan.ranks())
    off_o, sims_o, exact, lo, hi = oev.rank_bands(c, i, z, c, i, z, gap=1e-5, redux=redux, q_len=lens, c_len=lens)
    assert torch.equal(off_g, off_o)
    r = ranks_g.long()
    assert float((sims_g.double() - sims_o).abs().max()) <= 4e-6
    assert bool(((r >= lo) & (r <= hi)).all()), "a relevant item's rank left the band its 1e-5 neighbours allow"
    single = lo == hi
    assert torch.equal(r[single], exact[single])
    assert int(single.sum()) > 0.5 * single.numel()


@pytest.mark.parametrize("redux", REDUX)
@pytest.mark.parametrize("n,d", [(260, 64), (230, 96), (300, 48)])
def test_s32_all_vs_all_parity_with_oracle(n, d, redux):
    from wealy_b200 import evaluation as we
    c, i, z = _chunked_set(n, S, d, seed=n + d)
    aps_o, r1_o = oev.evaluate_argsort(c, i, z, c, i, z, redux=redux)
    cq, iq, zq = c.cuda(), i.cuda(), z.cuda()
    plan = we.EvalPlan(cq, iq, cq, iq)
    res = plan.run(zq, zq, redux=redux)
    torch.cuda.synchronize()
    aps, r1s = res["aps"].cpu().double(), res["r1s"].cpu().double()
    assert abs(float(aps.mean()) - float(aps_o.mean())) <= 1e-4
    assert abs(float(r1s.mean()) - float(r1_o.mean())) <= 1e-4 * max(1.0, float(r1_o.mean()))
    exact, _ = _check_r1(r1s, c, i, z, redux)
    assert torch.equal(r1s[exact], r1_o[exact])
    if redux in HALF:
        _check_all_item_ranks(plan, c, i, z, redux)
    plan.close()


@pytest.mark.parametrize("ragged", [False, True])
@pytest.mark.parametrize("redux", HALF)
def test_s32_half_sweep_equals_rectangle(redux, ragged, monkeypatch):
    """min / max reduce the same 1024 numbers in both sweeps (identical AP / R1); the mean's summation order differs
    between the half sweep's two directions (MAP within 1e-6)."""
    from wealy_b200 import evaluation as we
    n, d = 280, 64
    c, i, z = _chunked_set(n, S, d, seed=41)
    kw = {}
    if ragged:
        lens = _lens_spanning(n, seed=41)
        z = _pad_with_junk(z, lens, c, seed=41)
        kw = dict(q_chunks=lens, c_chunks=lens)
    cq, iq, zq = c.cuda(), i.cuda(), z.cuda()
    a1, r1 = we.evaluate(cq, iq, zq, cq, iq, zq, redux=redux, **kw)
    monkeypatch.setenv("WEALY_SYM_TRACKS", "0")
    a0, r0 = we.evaluate(cq, iq, zq, cq, iq, zq, redux=redux, **kw)
    if redux != "mean":
        assert torch.equal(a1, a0) and torch.equal(r1, r0)
    else:
        assert abs(float(a1.double().mean()) - float(a0.double().mean())) <= 1e-6


@pytest.mark.parametrize("redux", REDUX)
def test_s32_ragged_parity_with_oracle(redux):
    """Valid chunk counts 1 .. 32 (1, 16, 17 and 32 among them); the padding rows hold junk that would change every
    reduction if it were not excluded."""
    from wealy_b200 import evaluation as we
    n, d = 250, 64
    c, i, z = _chunked_set(n, S, d, seed=57)
    lens = _lens_spanning(n, seed=57)
    z = _pad_with_junk(z, lens, c, seed=58)
    aps_o, r1_o = oev.evaluate_argsort(c, i, z, c, i, z, redux=redux, q_len=lens, c_len=lens)
    cq, iq, zq = c.cuda(), i.cuda(), z.cuda()
    plan = we.EvalPlan(cq, iq, cq, iq)
    res = plan.run(zq, zq, redux=redux, q_chunks=lens, c_chunks=lens)
    torch.cuda.synchronize()
    aps, r1s = res["aps"].cpu().double(), res["r1s"].cpu().double()
    assert abs(float(aps.mean()) - float(aps_o.mean())) <= 1e-4
    assert abs(float(r1s.mean()) - float(r1_o.mean())) <= 1e-4 * max(1.0, float(r1_o.mean()))
    exact, _ = _check_r1(r1s, c, i, z, redux, lens)
    assert torch.equal(r1s[exact], r1_o[exact])
    if redux in HALF:
        _check_all_item_ranks(plan, c, i, z, redux, lens)
    plan.close()


@pytest.mark.parametrize("ragged", [False, True])
@pytest.mark.parametrize("redux", REDUX)
def test_s16_set_embedded_in_s32_matches_the_s16_path(redux, ragged):
    """An s = 16 set (full, or ragged with 1 .. 16 valid chunks) embedded in s = 32 with 16 junk padding rows per track
    and counts <= 16: min / max pick the same chunk similarities as the s = 16 kernels (identical AP / R1); the means
    divide in a different order (MAP within 1e-6).  Pins the 32-chunk K_pos layout and sweep to the s = 16 path."""
    from wealy_b200 import evaluation as we
    n, d = 200, 48
    c, i, z16 = _chunked_set(n, 16, d, seed=63)
    lens = torch.randint(1, 17, (n,), generator=torch.Generator().manual_seed(64)) if ragged else torch.full((n,), 16)
    z32 = torch.cat([z16, torch.zeros(n, 16, d)], dim=1)
    z32 = _pad_with_junk(z32, lens, c, seed=65)
    z16 = z32[:, :16].contiguous()
    cq, iq = c.cuda(), i.cuda()
    kw16 = dict(q_chunks=lens, c_chunks=lens) if ragged else {}
    for same in (True, False):
        if same:
            zg16, zg32 = z16.cuda(), z32.cuda()                    # one tensor on both sides: the half sweep
            a16, r16 = we.evaluate(cq, iq, zg16, cq, iq, zg16, redux=redux, **kw16)
            a32, r32 = we.evaluate(cq, iq, zg32, cq, iq, zg32, redux=redux, q_chunks=lens, c_chunks=lens)
        else:
            # queries != corpus: the rectangle sweep and K_pos on two operand sets
            cand = slice(60, n)
            sel = torch.tensor([t for t in range(60) if bool((c[cand] == c[t]).any())])
            qc, qi, cc, ci = cq[sel], iq[sel], cq[cand], iq[cand]
            kq = dict(q_chunks=lens[sel], c_chunks=lens[cand])
            a16, r16 = we.evaluate(qc, qi, z16[sel].cuda(), cc, ci, z16[cand].cuda(), redux=redux,
                                   **(kq if ragged else {}))
            a32, r32 = we.evaluate(qc, qi, z32[sel].cuda(), cc, ci, z32[cand].cuda(), redux=redux, **kq)
        if redux in ("min", "max"):
            assert torch.equal(a32, a16) and torch.equal(r32, r16)
        else:
            assert abs(float(a32.double().mean()) - float(a16.double().mean())) <= 1e-6


@pytest.mark.parametrize("redux", ["min", "meanmin", "mean"])
def test_s32_topk_queries_disjoint_from_corpus(redux):
    from wealy_b200 import evaluation as we
    n, d, k = 300, 64, 10
    c, i, z = _chunked_set(n, S, d, seed=71)
    q, cand = slice(0, 80), slice(80, n)
    keep = torch.tensor([bool((c[cand] == c[t]).any()) for t in range(80)])
    qc, qi, qz = c[q][keep], i[q][keep], z[q][keep].contiguous()
    aps_o, r1_o, idx_o, sim_o = oev.evaluate_argsort(qc, qi, qz, c[cand], i[cand], z[cand], topk=k, redux=redux)
    aps, r1s, idx, sim = we.evaluate(qc.cuda(), qi.cuda(), qz.cuda(), c[cand].cuda(), i[cand].cuda(), z[cand].cuda(),
                                     topk=k, redux=redux)
    idx, sim = idx.cpu(), sim.cpu()
    assert (sim - sim_o).abs().max() <= 4e-6
    ok = torch.ones_like(idx_o, dtype=torch.bool)
    ok[:, 1:] &= (sim_o[:, :-1] - sim_o[:, 1:]) > 1e-5
    ok[:, :-1] &= (sim_o[:, :-1] - sim_o[:, 1:]) > 1e-5
    ok[:, -1] = False   # the last position also depends on the (k+1)-th best, which the lists do not show
    assert torch.equal(idx[ok], idx_o[ok])
    assert abs(float(aps.double().mean().cpu()) - float(aps_o.mean())) <= 1e-4


def _emulated(c, i, z, world, redux, lens, staged):
    """Ranks 0 .. world-1 one after the other on plans of their own, counters (and, staged, thresholds) summed by hand
    where a multi-GPU run all-reduces them.  z is the flat [N * 32, D] layout (chunks=32)."""
    from wealy_b200 import evaluation as we
    plans = [we.EvalPlan(c, i, c, i) for _ in range(world)]
    thr = None
    if staged:
        for r, pl in enumerate(plans):
            pl.shard_prepare(z, r, world, redux=redux, q_chunks=lens, chunks=S)
            t = pl.thresholds_tensor()
            thr = t.clone() if thr is None else thr + t
        for pl in plans:
            pl.thresholds_tensor().copy_(thr)
    total = None
    for r, pl in enumerate(plans):
        if staged:
            pl.shard_sweep(r, world)
        else:
            pl.sweep_shard(z, r, world, redux=redux, q_chunks=lens, chunks=S)
        cnt = pl.counts_tensor()
        total = cnt.clone() if total is None else total + cnt
    plans[0].counts_tensor().copy_(total)
    out = plans[0].finish()
    torch.cuda.synchronize()
    return out, plans, thr


@pytest.mark.parametrize("staged", [False, True])
@pytest.mark.parametrize("ragged", [False, True])
@pytest.mark.parametrize("redux", ["min", "mean", "meanmin"])
def test_s32_sharded_sweep_emulated_on_one_gpu(redux, ragged, staged):
    """3 ranks: sweep_shard(..., chunks=32), or shard_prepare + shard_sweep; the summed counters give the single-GPU AP /
    R1 exactly, and the staged thresholds are the single-GPU K_pos bit for bit."""
    from wealy_b200 import evaluation as we
    n, d, world = 170, 64, 3
    c, i, z = _chunked_set(n, S, d, seed=83)
    lens = None
    if ragged:
        lens = _lens_spanning(n, seed=83)
        z = _pad_with_junk(z, lens, c, seed=84)
    cq, iq, zq = c.cuda(), i.cuda(), z.cuda()
    ref_plan = we.EvalPlan(cq, iq, cq, iq)
    ref = ref_plan.run(zq, zq, redux=redux, q_chunks=lens)
    out, plans, thr = _emulated(cq, iq, zq.reshape(n * S, d), world, redux, lens, staged)
    assert torch.equal(out["aps"], ref["aps"]) and torch.equal(out["r1s"], ref["r1s"])
    assert torch.allclose(out["sums"], ref["sums"], rtol=1e-9)
    if staged:
        m = max(ref_plan.total_pairs, 1)
        assert torch.equal(thr.view(torch.int32), ref_plan.thresholds_tensor()[-m:].view(torch.int32))
    for pl in plans:
        pl.close()
    ref_plan.close()


def test_s32_eval_pipeline_request():
    from wealy_b200 import evaluation as we
    n, d = 240, 64
    c, i, z = _chunked_set(n, S, d, seed=91)
    pipe = we.EvalPipeline(redux="max")
    t = pipe.submit(c, i, z.pin_memory())
    aps, r1s = pipe.result(t)
    aps, r1s = aps.clone(), r1s.clone()
    pipe.close()
    cq, iq, zq = c.cuda(), i.cuda(), z.cuda()
    a0, r0 = we.evaluate(cq, iq, zq, cq, iq, zq, redux="max")
    assert torch.equal(aps, a0.cpu()) and torch.equal(r1s, r0.cpu())
    aps_o, _ = oev.evaluate_argsort(c, i, z, c, i, z, redux="max")
    assert abs(float(aps.double().mean()) - float(aps_o.mean())) <= 1e-4


def test_s64_is_refused_on_every_entry():
    from wealy_b200 import dist as wd, evaluation as we
    n, d = 40, 32
    c, i, z = _chunked_set(n, 64, d, seed=97)
    cq, iq, zq = c.cuda(), i.cuda(), z.cuda()
    with pytest.raises(NotImplementedError):
        we.evaluate(cq, iq, zq, cq, iq, zq, redux="min")
    plan = we.EvalPlan(cq, iq, cq, iq)
    with pytest.raises(NotImplementedError):
        plan.sweep_shard(zq, 0, 2, redux="min")
    with pytest.raises(NotImplementedError):
        plan.sweep_shard(zq.reshape(n * 64, d), 0, 2, redux="min", chunks=64)
    with pytest.raises(NotImplementedError):
        wd._chunks_per_track(zq, None, "min", None)
    # the C ABI refuses 64 by itself (whole run and sharded sweep), before any work
    from wealy_b200 import _native as N
    zf = zq.reshape(n * 64, d)
    out = torch.empty(2 * n + 8, dtype=torch.float32, device="cuda")
    sums = torch.empty(3, dtype=torch.float64, device="cuda")
    with pytest.raises(NotImplementedError):
        N.check(N.lib.wealy_eval_run_chunked(plan._handle, zf.data_ptr(), d, zf.data_ptr(), d, d, N.F32, 1e-6, 3, 0, 64,
                                             N.REDUX["min"], out.data_ptr(), out[n:].data_ptr(), sums.data_ptr(), None,
                                             None, N.stream_ptr(zq.device)))
    with pytest.raises(NotImplementedError):
        N.check(N.lib.wealy_eval_sweep_shard_tracks(plan._handle, zf.data_ptr(), d, d, N.F32, 1e-6, 3, 64,
                                                    N.REDUX["min"], None, 0, 2, N.stream_ptr(zq.device)))
    torch.cuda.synchronize()
    plan.close()
