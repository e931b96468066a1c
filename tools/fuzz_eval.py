"""Randomised parity sweep of the evaluation paths against the oracle: random sizes / dims / dtypes / chunk counts /
reductions / clique structures; every relevant item's rank must lie in its 1e-5 band and be exact where the band is a
single rank.  Prints one JSON line.  Usage: python tools/fuzz_eval.py [seconds] [seed]"""
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


def one_case(rng, k):
    chunks = rng.choice([1, 1, 1, 2, 4, 8, 16, 32])
    n = rng.randint(260, 5000) if chunks == 1 else rng.randint(max(40, 300 // chunks), 2400 // chunks * 2)
    d = rng.choice([24, 48, 64, 100, 128, 200, 256, 333, 512, 1024])
    dtype = rng.choice([torch.float32, torch.float32, torch.float16, torch.bfloat16])
    sigma = rng.choice([None, 1.0, 2.5, 4.0])
    s = synth.make_eval_set(n, d, seed=1000 + k, **({"sigma": sigma} if sigma else {}))
    c, i, z = s["c"], s["i"], s["z"]
    redux = None
    lens = None
    if chunks > 1:
        g = torch.Generator().manual_seed(k)
        z = (z[:, None, :] + rng.choice([0.2, 0.8]) * z.norm(dim=1).mean() / d ** 0.5 * torch.randn(n, chunks, d, generator=g)).contiguous()
        redux = rng.choice(["min", "max", "mean", "meanmin", "minmean"])
        if rng.random() < 0.3:
            lens = torch.randint(1, chunks + 1, (n,), generator=g)
    z = z.to(dtype).float() if dtype != torch.float32 else z      # the oracle sees exactly the values the GPU gets
    same = rng.random() < 0.75
    kw = {}
    if redux:
        kw["redux"] = redux
    if lens is not None:
        kw["q_chunks"] = kw["c_chunks"] = lens
    zg = z.to(dtype).cuda()
    cg, ig = c.cuda(), i.cuda()
    if same:
        plan = we.EvalPlan(cg, ig, cg, ig)
        plan.run(zg, zg, **kw)
        qsel = torch.arange(n)
        cq, iq, zq, cc, ic, zc = c, i, z, c, i, z
        lq = lc = lens
    else:
        cut = n // 3
        qc_all, cand = slice(0, cut), slice(cut, n)
        keep = torch.tensor([bool(((c[cand] == c[t]) & (i[cand] != i[t])).any()) for t in range(cut)])
        if int(keep.sum()) < 2:
            return None
        cq, iq, zq = c[qc_all][keep], i[qc_all][keep], z[qc_all][keep]
        cc, ic, zc = c[cand], i[cand], z[cand]
        lq = lens[qc_all][keep] if lens is not None else None
        lc = lens[cand] if lens is not None else None
        kw2 = dict(kw)
        if lens is not None:
            kw2["q_chunks"], kw2["c_chunks"] = lq, lc
        plan = we.EvalPlan(cq.cuda(), iq.cuda(), cc.cuda(), ic.cuda())
        plan.run(zq.to(dtype).cuda(), zc.to(dtype).cuda(), **kw2)
    torch.cuda.synchronize()
    off_g, ranks_g, sims_g = (t.cpu() for t in plan.ranks())
    plan.close()
    off_o, sims_o, exact, lo, hi = oev.rank_bands(cq, iq, zq.double(), cc, ic, zc.double(), gap=1e-5, redux=redux, q_len=lq, c_len=lc)
    r = ranks_g.long()
    bad_off = not torch.equal(off_g, off_o)
    oob = int(((r < lo) | (r > hi)).sum()) if not bad_off else -1
    single = lo == hi
    mism = int((r[single] != exact[single]).sum()) if not bad_off else -1
    dsim = float((sims_g.double() - sims_o).abs().max()) if not bad_off and r.numel() else 0.0
    return {"n": n, "d": d, "chunks": chunks, "dtype": str(dtype).split(".")[-1], "sigma": sigma, "redux": redux,
            "ragged": lens is not None, "same": same, "items": int(r.numel()), "out_of_band": oob, "exact_mismatches": mism,
            "max_dsim": dsim, "offsets_differ": bad_off}


def main():
    budget = float(sys.argv[1]) if len(sys.argv) > 1 else 150.0
    seed = int(sys.argv[2]) if len(sys.argv) > 2 else 0
    rng = random.Random(seed)
    t0 = time.time()
    cases, bad, large = 0, [], []
    items = 0
    worst = 0.0
    k = 0
    while time.time() - t0 < budget:
        k += 1
        rec = one_case(rng, seed * 100000 + k)
        if rec is None:
            continue
        cases += 1
        items += rec["items"]
        worst = max(worst, rec["max_dsim"])
        if rec["out_of_band"] or rec["exact_mismatches"] or rec["offsets_differ"] or rec["max_dsim"] > 1e-5:
            bad.append(rec)
        elif rec["max_dsim"] > 5e-6:
            large.append(rec)      # beyond gap / 2 (where the band property is guaranteed a priori) yet inside the band
    print(json.dumps({"seed": seed, "seconds": round(time.time() - t0, 1), "cases": cases, "relevant_items_checked": items,
                      "max_abs_dsim_relevant_vs_float64": worst, "failing_cases": bad,
                      "cases_with_dsim_above_5e-6": large}), flush=True)


if __name__ == "__main__":
    main()
