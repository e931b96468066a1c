"""Multi-GPU evaluation of chunked tracks (SURVEY.md 8(f) rows e x f1): one JSON line.

--emulate W1,W2,..  (one GPU): for every world size W, each rank's share of the row-block-sharded chunked sweep is run
    in sequence on the one device -- plan.last_sweep_ms() (CUDA events around the sweep kernel) per rank after warm-up,
    median over --reps --; reported with the slowest / mean share, the sum of the shares against the unsharded sweep,
    and K_pos replicated on every rank (stage_ms()["kpos"] of the unsharded run) against the largest staged share
    (shard_prepare + shard_sweep of each rank: its share of the relevant track similarities plus the rebuild of the
    per-query limits; the float all-reduce between them needs several GPUs and is not measured here).
    Shapes: --shapes N x s x D list, min and mean, fp16x3 (the library default).

under `python -m torch.distributed.run --nproc-per-node N tools/dist_chunked_bench.py`: evaluate_all_vs_all end to end
    from pinned host memory and from resident device tensors, ms = max over the ranks of the host wall clock around
    --reps evaluations ending in a device synchronise; rank 0 checks the R1 of a 64-query sample against the oracle's
    rank bands.

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


def tracks(n, s, d, seed, device):
    """Chunk embeddings = the track's embedding + chunk-level noise (as tools/chunked_bench.py)."""
    base = synth.make_eval_set(n, d, seed=seed, device=device, md5_ids=False)
    g = torch.Generator(device=device).manual_seed(100 + seed)
    z = base["z"][:, None, :] + 0.8 * base["z"].norm(dim=1).mean() / d ** 0.5 * torch.randn(n, s, d, generator=g,
                                                                                            device=device)
    return base["c"], base["i"], z.contiguous()


def median_of(fn, reps):
    vals = []
    for _ in range(reps):
        vals.append(fn())
    return statistics.median(vals)


def emulate(args):
    worlds = [int(w) for w in args.emulate.split(",")]
    rec = {"mode": "emulate", "worlds": worlds, "reps": args.reps, "precision": "fp16x3", **gpu_info(), "cases": {}}
    for shape in args.shapes.split(","):
        n, s, d = (int(v) for v in shape.split("x"))
        c, i, z = tracks(n, s, d, seed=s, device="cuda")
        plan = we.EvalPlan(c, i, c, i)
        for redux in ("min", "mean"):
            def full():
                plan.run(z, z, redux=redux, allow_empty=True)
                st = plan.stage_ms()
                return plan.last_sweep_ms(), st["kpos"]
            for _ in range(2):
                full()
            runs = [full() for _ in range(args.reps)]
            sweep_ms = statistics.median(r[0] for r in runs)
            kpos_ms = statistics.median(r[1] for r in runs)
            case = {"unsharded_sweep_ms": sweep_ms, "kpos_replicated_ms": kpos_ms, "worlds": {}}
            for w in worlds:
                def share(r):
                    plan.sweep_shard(z, r, w, redux=redux)
                    return plan.last_sweep_ms()

                def staged(r):
                    plan.shard_prepare(z, r, w, redux=redux)
                    plan.shard_sweep(r, w)
                    return plan.stage_ms()["kpos"]
                for r in range(w):
                    share(r)
                    staged(r)
                per_rank = [median_of(lambda: share(r), args.reps) for r in range(w)]
                kpos_share = [median_of(lambda: staged(r), args.reps) for r in range(w)]
                mean = sum(per_rank) / w
                case["worlds"][str(w)] = {
                    "per_rank_sweep_ms": [round(v, 4) for v in per_rank],
                    "max_over_mean": max(per_rank) / mean,
                    "sum_over_unsharded": sum(per_rank) / sweep_ms,
                    "kpos_staged_share_ms": [round(v, 4) for v in kpos_share],
                    "kpos_staged_max_over_replicated": max(kpos_share) / kpos_ms,
                    "threshold_allreduce_bytes": 4 * max(plan.total_pairs, 1),
                }
            rec["cases"][f"{n}x{s}x{d}_{redux}"] = case
        plan.close()
        del z, c, i
        torch.cuda.empty_cache()
    return rec


def distributed(args):
    import torch.distributed as dist
    from oracle import evaluator as oev
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    rank, world = dist.get_rank(), dist.get_world_size()
    n, s, d = (int(v) for v in args.shapes.split(",")[0].split("x"))
    c, i, z = tracks(n, s, d, seed=s, device="cpu")               # the same set on every rank (seeded)
    z_pin = z.pin_memory()
    z_dev = z.to(dev)
    rec = {"mode": "distributed", "world": world, "shape": [n, s, d], "precision": "fp16x3", "reps": args.reps,
           **gpu_info(), "runs": {}}
    for redux in ("min", "mean"):
        for label, zin in (("pinned_host", z_pin), ("resident", z_dev)):
            def step():
                out = wd.evaluate_all_vs_all(c, i, zin, redux=redux)
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
            ms = float(t.item())
            rec["runs"][f"{redux}_{label}"] = {"ms": ms, "track_pairs_per_s": n * n / (ms * 1e-3),
                                                "chunk_pairs_per_s": (n * s) ** 2 / (ms * 1e-3), "map": out["map"]}
        if rank == 0:
            qs = torch.randperm(n, generator=torch.Generator().manual_seed(1))[:64]
            lo, hi = oev.rank_tolerance(c[qs], i[qs], z[qs], c, i, z, gap=1e-5, redux=redux)
            r1 = out["r1s"].cpu().double()[qs]
            ok = bool(((r1 >= lo) & (r1 <= hi)).all())
            rec["runs"][f"{redux}_parity64"] = {"r1_inside_bands": ok, "exact_bands": int((lo == hi).sum()),
                                                "r1_exact_where_single": bool(torch.equal(r1[lo == hi], lo[lo == hi]))}
    dist.destroy_process_group()
    return rec if rank == 0 else None


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--emulate", default=None, help="comma-separated world sizes, ranks run in sequence on one GPU")
    ap.add_argument("--shapes", default="12500x8x1024,50000x8x1024", help="N x s x D, comma-separated")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the record to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("dist_chunked_bench.py measures on a CUDA device; none is available")
    rec = emulate(args) if args.emulate else distributed(args)
    if rec is not None:
        line = json.dumps(rec)
        print(line, flush=True)
        if args.out:
            with open(args.out, "w") as f:
                f.write(line + "\n")


if __name__ == "__main__":
    main()
