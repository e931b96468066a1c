"""The symmetric sweep's threshold-level variants count the same ranks.

The epilogue scores clean tiles by counting compares and dirty tiles with bit masks; how many levels are handled
densely (WEALY_SYM_LEVELS) and which core runs it (WEALY_SYM_PAIR=0: single CTA) change only how the rank counters
are reached.  Every variant must return the default's per-query AP and R1 bit for bit, on easy and on hard data."""
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("sigma", [1.5, 3.5])
def test_level_and_core_variants_match_the_default(monkeypatch, sigma):
    from wealy_b200 import evaluation as we
    from wealy_b200.data import synth
    s = synth.make_eval_set(6000, 256, seed=7, sigma=sigma)
    c, i, z = s["c"].cuda(), s["i"].cuda(), s["z"].cuda()

    def run():
        plan = we.EvalPlan(c, i, c, i)
        res = plan.run(z, z)
        out = res["aps"].clone(), res["r1s"].clone()
        plan.close()
        return out

    aps0, r1s0 = run()
    assert float(aps0.double().mean()) > 0.0
    for pair in ("1", "0"):
        for lv in ("2", "3", "4"):
            monkeypatch.setenv("WEALY_SYM_PAIR", pair)
            monkeypatch.setenv("WEALY_SYM_LEVELS", lv)
            aps, r1s = run()
            assert torch.equal(aps, aps0) and torch.equal(r1s, r1s0), (pair, lv)
