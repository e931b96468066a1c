"""Timing of the rectangle sweeps (everything that is not the symmetric all-vs-all sweep): queries != corpus, chunked
tracks, all-vs-all top-k forced onto the streaming path.  Prints one JSON line."""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import wealy_b200  # noqa: E402,F401
from wealy_b200 import evaluation as we  # noqa: E402
from wealy_b200.data import synth  # noqa: E402


def timed(fn, warm=2, reps=4):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        r = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps, r


def main():
    out = {}
    s = synth.make_eval_set(200_000, 1024, seed=0, device="cuda", md5_ids=False)
    q, c = slice(0, 100_000), slice(100_000, 200_000)
    keep = torch.isin(s["c"][q], s["c"][c])               # queries with a relevant item in the corpus half
    qc, qi, qz = s["c"][q][keep], s["i"][q][keep], s["z"][q][keep].contiguous()
    plan = we.EvalPlan(qc, qi, s["c"][c], s["i"][c])
    cz = s["z"][c].contiguous()
    ms, r = timed(lambda: plan.run(qz, cz))
    out["queries_vs_corpus"] = {"nq": int(qc.numel()), "nc": 100_000, "ms": ms, "gpairs_per_s": qc.numel() * 1e5 / (ms * 1e-3) / 1e9,
                                "sweep_ms": plan.last_sweep_ms(), "map": float(r["sums"][0] / r["sums"][2])}
    plan.close()
    del s, plan
    torch.cuda.empty_cache()
    n, ch = 12_500, 8
    s = synth.make_eval_set(n * ch, 1024, seed=1, device="cuda", md5_ids=False)
    ids = synth.make_eval_set(n, 8, seed=2, device="cuda", md5_ids=False)
    z = s["z"].view(n, ch, 1024)
    plan = we.EvalPlan(ids["c"], ids["i"], ids["c"], ids["i"])
    for label, env in (("chunked_tracks", "1"), ("chunked_tracks_rectangle", "0")):   # half sweep (default) / full rectangle
        os.environ["WEALY_SYM_TRACKS"] = env
        ms, r = timed(lambda: plan.run(z, z, redux="min", allow_empty=True))
        out[label] = {"tracks": n, "chunks": ch, "ms": ms, "g_chunk_pairs_per_s": (n * ch) ** 2 / (ms * 1e-3) / 1e9,
                      "sweep_ms": plan.last_sweep_ms(), "map": float(r["sums"][0] / r["sums"][2])}
    plan.close()
    # 2 chunks per track: a quarter of the elements survive the reduction (the column direction's worst case)
    n2 = 50_000
    ids2 = synth.make_eval_set(n2, 8, seed=3, device="cuda", md5_ids=False)
    z2 = s["z"].view(n2, 2, 1024)
    plan = we.EvalPlan(ids2["c"], ids2["i"], ids2["c"], ids2["i"])
    for label, env in (("chunked_2", "1"), ("chunked_2_rectangle", "0")):
        os.environ["WEALY_SYM_TRACKS"] = env
        ms, r = timed(lambda: plan.run(z2, z2, redux="mean", allow_empty=True))
        out[label] = {"tracks": n2, "chunks": 2, "redux": "mean", "ms": ms, "sweep_ms": plan.last_sweep_ms(),
                      "map": float(r["sums"][0] / r["sums"][2])}
    os.environ.pop("WEALY_SYM_TRACKS")
    plan.close()
    del z2
    del s, plan, z
    torch.cuda.empty_cache()
    os.environ["WEALY_SYM_TOPK"] = "0"
    s = synth.make_eval_set(50_000, 2048, seed=5, dist="lyric_covers_test", device="cuda", md5_ids=False)
    plan = we.EvalPlan(s["c"], s["i"], s["c"], s["i"])
    ms, r = timed(lambda: plan.run(s["z"], s["z"], topk=100))
    out["c5_rect_topk100"] = {"ms": ms, "sweep_ms": plan.last_sweep_ms(), "path": plan.last_topk_path()}
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
