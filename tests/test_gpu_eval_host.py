"""-m gpu: wealy_eval_run_host (pinned host embeddings read by the device while the symmetric sweep runs) must give
exactly what wealy_eval_run gives on a device copy -- same planes bit for bit, so the same counters, AP and R1."""
import os

import pytest
import torch

from oracle import evaluator as oev

pytestmark = pytest.mark.gpu


def _we():
    from wealy_b200 import evaluation as we
    return we


def _synth():
    from wealy_b200.data import synth
    return synth


def _both(c, i, z, **kw):
    we = _we()
    cd, idd = c.cuda(), i.cuda()
    plan = we.EvalPlan(cd, idd, cd, idd)
    try:
        zd = z.cuda()
        ref = plan.run(zd, zd, **kw)
        ref_ranks = [t.cpu() for t in plan.ranks()]
        ref = {k: v.cpu() for k, v in ref.items()}
        zh = z.pin_memory()
        got = plan.run_host(zh, **kw)
        got_ranks = [t.cpu() for t in plan.ranks()]
        got = {k: v.cpu() for k, v in got.items()}
        torch.cuda.synchronize()
    finally:
        plan.close()
    return ref, got, ref_ranks, got_ranks


def _assert_same(ref, got, ref_ranks, got_ranks):
    # (queries without a relevant item score NaN on both routes)
    assert torch.equal(ref["aps"].isnan(), got["aps"].isnan())
    assert torch.equal(ref["aps"].nan_to_num(-1.0), got["aps"].nan_to_num(-1.0)), float((ref["aps"] - got["aps"]).abs().nan_to_num(0).max())
    assert torch.equal(ref["r1s"].nan_to_num(-1.0), got["r1s"].nan_to_num(-1.0))
    assert torch.equal(ref["sums"], got["sums"])
    for a, b in zip(ref_ranks, got_ranks):
        assert torch.equal(a, b)


@pytest.mark.parametrize("n,d", [(5, 8), (300, 64), (1500, 256), (7001, 128), (9000, 1024), (26000, 64)])
def test_host_run_is_bit_identical_to_the_device_run(n, d):
    s = _synth().make_eval_set(n, d, seed=n) if n > 16 else None
    if s is None:
        z = torch.randn(n, d)
        c = torch.tensor([0, 0, 1, 1, 1]); i = torch.arange(n)
    else:
        z, c, i = s["z"], s["c"], s["i"]
    _assert_same(*_both(c, i, z))


@pytest.mark.parametrize("parts", [1, 2, 5, 7])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float16, torch.bfloat16])
def test_every_part_schedule_and_dtype(parts, dtype, monkeypatch):
    monkeypatch.setenv("WEALY_HOST_PARTS", str(parts))
    s = _synth().make_eval_set(6000, 96, seed=3)
    _assert_same(*_both(s["c"], s["i"], s["z"].to(dtype)))


@pytest.mark.parametrize("clique", [359, 1100])
def test_cliques_that_straddle_part_boundaries(clique, monkeypatch):
    # K_pos of a part reads the rows of whole cliques: a giant clique reaches far below the part's first row block
    monkeypatch.setenv("WEALY_HOST_PARTS", "7")
    n, d = 8000, 64
    g = torch.Generator().manual_seed(clique)
    z = torch.randn(n, d, generator=g)
    c = torch.arange(n) // 2 + 10
    pos = torch.randperm(n, generator=g)[:clique]
    c[pos] = 5                                   # sorts FIRST: the giant clique sits where the last part begins
    c2 = c.clone()
    c2[pos] = int(c.max()) + 7                   # ... and the same clique sorting LAST
    i = torch.arange(n)
    for cc in (c, c2):
        ref, got, rr, gr = _both(cc, i, z, allow_empty=True)
        _assert_same(ref, got, rr, gr)


def test_single_pass_precision_and_oracle_parity():
    s = _synth().make_eval_set(3000, 128, seed=11)
    ref, got, rr, gr = _both(s["c"], s["i"], s["z"], precision="fp16")
    _assert_same(ref, got, rr, gr)
    # ... and the 3-pass host run against the float64 oracle's rank bands
    ref, got, rr, gr = _both(s["c"], s["i"], s["z"])
    off_o, _, exact, lo, hi = oev.rank_bands(s["c"], s["i"], s["z"], s["c"], s["i"], s["z"], gap=1e-5)
    off_g, ranks_g, _ = gr
    assert torch.equal(off_g, off_o)
    assert bool(((ranks_g.long() >= lo) & (ranks_g.long() <= hi)).all())
    assert torch.equal(ranks_g.long()[lo == hi], exact[lo == hi])


def test_evaluate_routes_pinned_host_tensors_through_the_pipeline(monkeypatch):
    we = _we()
    monkeypatch.setenv("WEALY_HOST_STREAM_MIN_ROWS", "1000")   # (the default routes sets of >= 24576 rows)
    s = _synth().make_eval_set(2500, 256, seed=5)
    c, i, z = s["c"], s["i"], s["z"]
    cd, idd, zd = c.cuda(), i.cuda(), z.cuda()
    aps_d, r1s_d = we.evaluate(cd, idd, zd, cd, idd, zd)
    assert we.last_path() == "device"
    zp = z.pin_memory()
    aps_h, r1s_h = we.evaluate(c, i, zp, c, i, zp)
    assert we.last_path() == "host_stream"
    assert torch.equal(aps_d.cpu(), aps_h.cpu()) and torch.equal(r1s_d.cpu(), r1s_h.cpu())
    # pageable memory, top-k, and the opt-out keep the copy-then-compute path (same numbers)
    aps_p, r1s_p = we.evaluate(c, i, z, c, i, z)
    assert we.last_path() == "device" and torch.equal(aps_p.cpu(), aps_d.cpu())
    res = we.evaluate(c, i, zp, c, i, zp, topk=5)
    assert we.last_path() == "device" and torch.equal(res[0].cpu(), aps_d.cpu())
    monkeypatch.setenv("WEALY_HOST_STREAM", "0")
    aps_o, _ = we.evaluate(c, i, zp, c, i, zp)
    assert we.last_path() == "device" and torch.equal(aps_o.cpu(), aps_d.cpu())


def test_host_run_refuses_what_it_cannot_read():
    we = _we()
    s = _synth().make_eval_set(400, 32, seed=1)
    cd, idd = s["c"].cuda(), s["i"].cuda()
    plan = we.EvalPlan(cd, idd, cd, idd)
    try:
        with pytest.raises(NotImplementedError):
            plan.run_host(s["z"].clone())                      # pageable
        with pytest.raises(NotImplementedError):
            plan.run_host(torch.randn(400, 30).pin_memory())   # rows of 30 elements
        with pytest.raises(NotImplementedError):
            plan.run_host(torch.randn(400, 2048).pin_memory())  # rows beyond 1024 elements
        got = plan.run_host(s["z"].cuda())                     # a device pointer takes the plain path
        zd = s["z"].cuda()
        ref = plan.run(zd, zd)
        assert torch.equal(got["aps"], ref["aps"])
    finally:
        plan.close()
    # a plan whose two sides differ is not an all-vs-all plan
    plan = we.EvalPlan(cd[:100], idd[:100], cd, idd)
    try:
        with pytest.raises((NotImplementedError, AssertionError)):
            plan.run_host(s["z"].pin_memory())
    finally:
        plan.close()


def test_default_threshold_keeps_small_sets_on_the_copy_engine():
    we = _we()
    s = _synth().make_eval_set(2500, 64, seed=5)
    zp = s["z"].pin_memory()
    we.evaluate(s["c"], s["i"], zp, s["c"], s["i"], zp)
    assert we.last_path() == "device"


@pytest.mark.parametrize("n,parts", [(3000, 1), (7000, 2), (6000, 5), (1000, 7)])
def test_early_upload_inside_the_plan_build(n, parts, monkeypatch):
    # wealy_eval_plan_create_host starts the upload of the first part under the plan build; the run fetches the rest.
    # (1000, 7): the first part is empty, so the padding rows belong to the second
    monkeypatch.setenv("WEALY_HOST_PARTS", str(parts))
    we = _we()
    s = _synth().make_eval_set(n, 128, seed=n)
    cd, idd, zd = s["c"].cuda(), s["i"].cuda(), s["z"].cuda()
    zp = s["z"].pin_memory()
    ref_plan = we.EvalPlan(cd, idd, cd, idd)
    ref = ref_plan.run(zd, zd)
    plan = we.EvalPlan(cd, idd, cd, idd, host_z=zp)
    got = plan.run_host(zp)
    assert torch.equal(ref["aps"], got["aps"]) and torch.equal(ref["r1s"], got["r1s"])
    # a run on OTHER embeddings ignores the early upload ...
    z2 = (s["z"] * 0.5 + 0.1).pin_memory()
    plan2 = we.EvalPlan(cd, idd, cd, idd, host_z=zp)
    got2 = plan2.run_host(z2)
    z2d = z2.cuda()
    ref2 = ref_plan.run(z2d, z2d)
    assert torch.equal(ref2["aps"], got2["aps"])
    # ... and so does the device route; a plan that is never run is torn down cleanly
    got3 = we.EvalPlan(cd, idd, cd, idd, host_z=zp).run(zd, zd)
    assert torch.equal(ref["aps"], got3["aps"])
    we.EvalPlan(cd, idd, cd, idd, host_z=zp).close()
    torch.cuda.synchronize()
    for pl in (ref_plan, plan, plan2):
        pl.close()
