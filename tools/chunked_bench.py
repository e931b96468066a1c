"""Chunked all-vs-all (SURVEY.md 8(f) row f1): half sweep (default) against the full rectangle (WEALY_SYM_TRACKS=0) on
track-structured data: chunk embeddings = the track's embedding + chunk-level noise.  Every shape has the same 100 000
chunk rows (so the same MMA work): 100 000 / s tracks x s chunks x 1024.  Per shape and reduction: the whole call (ms),
the sweep kernel and the stages of the last call (plan.stage_ms(), CUDA events), and the MAP.  --chunks picks the chunk
counts (default 2,4,8,16,32).  The GPU name and power limit are read in the same run.  One JSON line."""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import wealy_b200  # noqa: E402,F401
from wealy_b200 import evaluation as we  # noqa: E402
from wealy_b200.data import synth  # noqa: E402
from rect_bench import timed  # noqa: E402
from dist_chunked_bench import gpu_info  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--chunks", default="2,4,8,16,32")
    args = ap.parse_args()
    out = gpu_info()
    rows, d = 100_000, 1024
    for ch in (int(x) for x in args.chunks.split(",")):
        n = rows // ch
        base = synth.make_eval_set(n, d, seed=ch, device="cuda", md5_ids=False)
        g = torch.Generator(device="cuda").manual_seed(100 + ch)
        z = base["z"][:, None, :] + 0.8 * base["z"].norm(dim=1).mean() / d ** 0.5 * torch.randn(n, ch, d, generator=g, device="cuda")
        z = z.contiguous()
        plan = we.EvalPlan(base["c"], base["i"], base["c"], base["i"])
        for redux in ("min", "mean"):
            rec = {}
            for label, env in (("half", "1"), ("rectangle", "0")):
                os.environ["WEALY_SYM_TRACKS"] = env
                ms, r = timed(lambda: plan.run(z, z, redux=redux, allow_empty=True))
                rec[label] = {"ms": ms, "sweep_ms": plan.last_sweep_ms(), "stage_ms": plan.stage_ms(),
                              "map": float(r["sums"][0] / r["sums"][2])}
            out[f"{n}x{ch}_{redux}"] = rec
        plan.close()
        del z, base
        torch.cuda.empty_cache()
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
