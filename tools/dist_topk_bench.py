"""Multi-GPU all-vs-all top-k on the row-block-sharded symmetric sweep: one JSON line.

--emulate W1,W2,..  (one GPU), at BASELINE configs[4] by default (50 000 x 2048, top-100, fp16x3): for every world size
    W, each rank's call of EvalPlan.sweep_shard_topk is run in sequence on the one device.  Per rank: its share = the
    sweep over its row blocks + the local finalize (stage_ms() sweep + topk_finalize, CUDA events), median of --reps;
    reported with the slowest / mean share and the sum of the shares against the unsharded symmetric call's sweep +
    finalize (`sum_over_unsharded`) and against the whole unsharded call (`sum_over_unsharded_call`).  The part every
    rank repeats -- normalisation, relevant similarities, sampled pre-pass and bounds (stage_ms() prep + kpos) -- is
    reported on its own.  Also: the merge of rank 0's query slice (merge_topk on the
    lists of all ranks: CUDA events around the call, its 4-byte read-back included), the bytes each rank sends and
    receives in the list exchange and the all-gather of the merged slices, and the per-rank time of the
    query-partitioned path the sharded one replaces (rank 0's query slice against the whole corpus with the rectangle
    sweep's streaming top-k: CUDA events around plan.run, median of --reps).

under `python -m torch.distributed.run --nproc-per-node N tools/dist_topk_bench.py`: evaluate_all_vs_all(topk=k) end to
    end from resident device tensors, ms = max over the ranks of the host wall clock around --reps evaluations ending in
    a device synchronise, on the sharded route and (WEALY_SYM_TOPK=0) on the query-partitioned one.

The GPU name and power limit are read in the same run and written into the record."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import wealy_b200  # noqa: E402,F401
from wealy_b200 import evaluation as we, dist as wd  # noqa: E402
from wealy_b200.data import synth  # noqa: E402


def gpu_info():
    """Name and power limit of the device this process runs on (nvidia-smi query; read-only)."""
    idx = torch.cuda.current_device()
    out = {"gpu": torch.cuda.get_device_name(idx)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(idx), "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        out["power_limit_and_max_sm_clock"] = q
    except (OSError, subprocess.SubprocessError):
        out["power_limit_and_max_sm_clock"] = "unavailable"
    return out


def eval_set(n, d, device):
    """The configs[4] set: lyric-covers clique sizes (as tests/test_gpu_eval.py's configs[4] test)."""
    s = synth.make_eval_set(n, d, seed=5, dist="lyric_covers_test", device=device, md5_ids=False)
    return s["c"], s["i"], s["z"]


def event_ms(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1)


def emulate(args):
    worlds = [int(w) for w in args.emulate.split(",")]
    n, d, k = args.n, args.d, args.k
    c, i, z = eval_set(n, d, "cuda")
    plan = we.EvalPlan(c, i, c, i)
    rec = {"mode": "emulate", "shape": [n, d], "k": k, "precision": "fp16x3", "reps": args.reps, **gpu_info(),
           "worlds": {}}

    def full():
        plan.run(z, z, topk=k)
        assert plan.last_topk_path() == 1
        return plan.stage_ms()
    for _ in range(2):
        full()
    runs = [full() for _ in range(args.reps)]
    med = {key: statistics.median(r[key] for r in runs) for key in runs[0]}
    unsharded = med["sweep"] + med["topk_finalize"]
    rec["unsharded_stage_ms"] = {key: round(v, 4) for key, v in med.items()}
    rec["unsharded_sweep_plus_finalize_ms"] = unsharded
    rec["unsharded_call_ms"] = sum(med.values())
    for w in worlds:
        def share(r):
            loc = plan.sweep_shard_topk(z, r, w, k)
            st = plan.stage_ms()
            return st, loc
        for r in range(w):
            share(r)
        per_rank, fixed, locs = [], [], []
        for r in range(w):
            sts = []
            for _ in range(args.reps):
                st, loc = share(r)
                sts.append(st)
            locs.append(loc)
            per_rank.append(statistics.median(s["sweep"] + s["topk_finalize"] for s in sts))
            fixed.append(statistics.median(s["prep"] + s["kpos"] for s in sts))
        finalize = statistics.median(s["topk_finalize"] for s in sts)
        lo, hi = wd.shard_range(n, 0, w)
        val = torch.stack([l["val"][lo:hi] for l in locs])
        idx = torch.stack([l["idx"][lo:hi] for l in locs])
        cnt = torch.stack([l["cnt"][lo:hi] for l in locs])
        failed = [0]

        def merge():
            failed[0] = we.merge_topk(val, idx, cnt)[2]
        merge()
        merge_ms = statistics.median(event_ms(merge) for _ in range(args.reps))
        del locs, val, idx, cnt
        qplan = we.EvalPlan(c[lo:hi], i[lo:hi], c, i)
        zq = z[lo:hi]
        for _ in range(2):
            qplan.run(zq, z, topk=k)
        query_ms = statistics.median(event_ms(lambda: qplan.run(zq, z, topk=k)) for _ in range(args.reps))
        qplan.close()
        mean = sum(per_rank) / w
        row = 4 * (2 * k + 1)
        rec["worlds"][str(w)] = {
            "per_rank_share_ms": [round(v, 4) for v in per_rank],
            "max_over_mean": max(per_rank) / mean,
            "sum_over_unsharded": sum(per_rank) / unsharded,
            "sum_over_unsharded_call": sum(per_rank) / rec["unsharded_call_ms"],
            "replicated_prep_kpos_prepass_ms": round(statistics.median(fixed), 4),
            "local_finalize_ms_last_rank": round(finalize, 4),
            "per_rank_total_ms": round(max(per_rank) + statistics.median(fixed), 4),
            "merge_ms_rank0_slice": round(merge_ms, 4),
            "merge_failed_queries": failed[0],
            "exchange_bytes_sent_rank0": (n - (hi - lo)) * row,
            "exchange_bytes_received_rank0": (w - 1) * (hi - lo) * row,
            "gather_bytes_received_rank0": (n - (hi - lo)) * k * 12,
            "query_partitioned_rank0_ms": round(query_ms, 4),
        }
    plan.close()
    return rec


def distributed(args):
    import torch.distributed as dist
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    rank, world = dist.get_rank(), dist.get_world_size()
    c, i, z = eval_set(args.n, args.d, "cpu")                        # the same set on every rank (seeded)
    c, i, z = c.to(dev), i.to(dev), z.to(dev)
    rec = {"mode": "distributed", "world": world, "shape": [args.n, args.d], "k": args.k, "precision": "fp16x3",
           "reps": args.reps, **gpu_info(), "runs": {}}
    for label, env in (("sym_sharded", "1"), ("query_sharded", "0")):
        os.environ["WEALY_SYM_TOPK"] = env

        def step():
            out = wd.evaluate_all_vs_all(c, i, z, topk=args.k)
            out["plan"].close()
            return out
        for _ in range(2):
            out = step()
        torch.cuda.synchronize()
        dist.barrier()
        t0 = time.perf_counter()
        for _ in range(args.reps):
            out = step()
        torch.cuda.synchronize()
        t = torch.tensor([(time.perf_counter() - t0) * 1e3 / args.reps], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        rec["runs"][label] = {"ms": float(t.item()), "topk_path": out["topk_path"], "map": out["map"]}
    os.environ.pop("WEALY_SYM_TOPK")
    dist.destroy_process_group()
    return rec if rank == 0 else None


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--emulate", default=None, help="comma-separated world sizes, ranks run in sequence on one GPU")
    ap.add_argument("--n", type=int, default=50_000)
    ap.add_argument("--d", type=int, default=2048)
    ap.add_argument("--k", type=int, default=100)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the record to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("dist_topk_bench.py measures on a CUDA device; none is available")
    rec = emulate(args) if args.emulate else distributed(args)
    if rec is not None:
        line = json.dumps(rec)
        print(line, flush=True)
        if args.out:
            with open(args.out, "w") as f:
                f.write(line + "\n")


if __name__ == "__main__":
    main()
