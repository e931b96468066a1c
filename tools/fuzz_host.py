"""Randomised comparison of wealy_eval_run_host (pinned host embeddings, upload / prep / sweep pipeline) with wealy_eval_run
on a device copy: random sizes / dims / dtypes / row strides / clique structures / part schedules / early uploads.
AP, R1, the running sums and the rank of every relevant item must be IDENTICAL (the planes are bit-identical); every
tenth case is also held against the oracle's rank bands.  One JSON line.  Usage: python tools/fuzz_host.py [seconds] [seed]"""
import json
import os
import random
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import wealy_b200  # noqa: E402,F401
from oracle import evaluator as oev  # noqa: E402
from wealy_b200 import evaluation as we  # noqa: E402
from wealy_b200.data import synth  # noqa: E402


def same(a, b):
    return bool(torch.equal(a.isnan(), b.isnan()) and torch.equal(a.nan_to_num(-1.0), b.nan_to_num(-1.0)))


def main():
    budget = float(sys.argv[1]) if len(sys.argv) > 1 else 30.0
    seed = int(sys.argv[2]) if len(sys.argv) > 2 else 1
    rng = random.Random(seed)
    t0 = time.time()
    out = {"seed": seed, "cases": 0, "rows": 0, "relevant_items": 0, "mismatches": [], "oracle_cases": 0,
           "oracle_out_of_band": 0, "early_upload_cases": 0}
    k = 0
    while time.time() - t0 < budget:
        k += 1
        n = rng.choice([rng.randint(2, 300), rng.randint(300, 9000), rng.randint(9000, 40000)])
        d = 4 * rng.randint(1, 256) if rng.random() < 0.5 else rng.choice([64, 128, 256, 512, 1024])
        if n > 9000:
            d = min(d, 256)
        dtype = rng.choice([torch.float32, torch.float32, torch.float16, torch.bfloat16])
        parts = rng.choice([0, 1, 2, 5, 7])
        os.environ["WEALY_HOST_PARTS"] = str(parts)
        dist = rng.choice(["shs100k_test", "lyric_covers_test"])
        s = synth.make_eval_set(max(n, 4), d, seed=7000 + k, dist=dist, md5_ids=rng.random() < 0.5)
        c, i, z = s["c"], s["i"], s["z"].to(dtype)
        n = z.shape[0]
        if rng.random() < 0.3 and n > 600:   # one giant clique, somewhere in the sorted order
            g = torch.Generator().manual_seed(k)
            c = c.clone()
            c[torch.randperm(n, generator=g)[: rng.randint(200, min(2500, n // 2))]] = rng.choice([-5, int(c.max()) // 2, int(c.max()) + 9])
        pad = rng.choice([0, 0, 4, 12])      # row stride beyond d
        zh = torch.empty(n, d + pad, dtype=dtype).pin_memory()[:, :d]
        zh.copy_(z)
        cd, idd, zd = c.cuda(), i.cuda(), z.cuda()
        early = rng.random() < 0.5
        ref_plan = we.EvalPlan(cd, idd, cd, idd)
        ref = ref_plan.run(zd, zd, allow_empty=True)
        ref_ranks = ref_plan.ranks()
        plan = we.EvalPlan(cd, idd, cd, idd, host_z=zh if early else None)
        got = plan.run_host(zh, allow_empty=True)
        got_ranks = plan.ranks()
        ok = same(ref["aps"], got["aps"]) and same(ref["r1s"], got["r1s"]) and torch.equal(ref["sums"], got["sums"]) and \
            all(torch.equal(a, b) for a, b in zip(ref_ranks, got_ranks))
        out["cases"] += 1
        out["rows"] += n
        out["relevant_items"] += int(ref_plan.total_pairs)
        out["early_upload_cases"] += int(early)
        if not ok:
            out["mismatches"].append({"case": k, "n": n, "d": d, "dtype": str(dtype), "parts": parts, "early": early})
        if k % 10 == 0 and n <= 6000:
            zf = z.float()
            off_o, _, exact, lo, hi = oev.rank_bands(c, i, zf, c, i, zf, gap=1e-5)
            r = got_ranks[1].cpu().long()
            out["oracle_cases"] += 1
            out["oracle_out_of_band"] += int(((r < lo) | (r > hi)).sum()) + int((r[lo == hi] != exact[lo == hi]).sum())
        ref_plan.close()
        plan.close()
    out["seconds"] = time.time() - t0
    print(json.dumps(out))


if __name__ == "__main__":
    main()
