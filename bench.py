#!/usr/bin/env python
"""bench.py -- headline benchmark of the WEALY retrieval-and-scoring hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--precision fp16x3|fp16]
                    [--legs main,c1,c3,c4,c5,f1] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

Metric (BASELINE.json): similarity + MAP evaluation throughput in Gpairs/s, pairs = Nq * Nc per
evaluate.  One *step* = one full fused evaluation (prep -> relevant thresholds -> tcgen05 sweep with
mask / rank-count epilogue -> AP reduce -> MAP) of the workload:

  N = 1 : BASELINE.json configs[1] -- Discogs-VI-YT-test-shaped all-vs-all, 100 000 x 1024-d fp32
          synthetic embeddings, clique sizes bootstrapped from the shipped SHS100K-TEST split.
  N > 1 : the same all-vs-all grown so that every GPU keeps 1e10 pairs (weak scaling):
          N_total = 100 000 * sqrt(N) tracks, corpus replicated; every rank sweeps the row blocks
          rank (mod N) of the symmetric problem and the per-(query, relevant item) rank counters are
          summed with ONE NCCL all-reduce per step (the path's only exchange), after which every
          rank holds the complete AP / R1.

`value`  : whole-job Gpairs/s with embeddings and ids already resident in HBM (id-only plan built
           once, outside the timed region).
`e2e`    : the same metric through the public API `wealy_b200.evaluation.evaluate()` with HOST
           (pinned) buffers: every step pays the host->device copy of embeddings and ids, the plan
           build, the evaluation and the device->host read of per-query AP / R1.
`parity` : at every N, rank 0 scores a query sample with the CPU oracle and compares MAP / MR1, R1 and the
           rank of EVERY relevant item (bit-exact wherever the similarity gap exceeds 1e-5).

The other BASELINE.json configs ride on the same JSON line as extra keys (each a few steps):
  `c1_shs100k`  configs[0]: 10 547 x 1024 (the exact SHS100K-TEST clique multiset), GPU vs the FULL CPU run
  `c3_500k`     configs[2]: 500 000 x 1024 all-vs-all on the N GPUs of this run (strong-scaling series)
  `c4_loss`     configs[3]: NT-Xent / CLEWS forward + backward, batch 4096 x 1024 bf16 (N = 1 only)
  `c5_topk100`  configs[4]: 50 000 x 2048, top-100 output (N = 1 only)

`--impl reference`: the reference's CPU implementation of the path (it is pure Python / torch, so
           the timed code is the oracle port: torch matmul similarity + per-query argsort
           evaluator) on all host cores, on a bounded query sample of the same workload.  This arm
           never loads the CUDA library.

`--dump-outputs DIR`: after the timed steps, what the timed path returned in its last step goes to DIR/<name>.npy
           (float32 / float64): per-query `aps` and `r1s` and the `sums` {sum AP, sum R1, #scored}.  The inputs are
           seeded, so two builds run with the same arguments can be compared output for output: `aps` and `r1s`
           repeat bit for bit, while sum AP is a float64 reduction on the device whose last bits vary from run to run.

The benchmark writes nothing into the tree it runs from (which may be read-only).
"""
import argparse
import importlib.util
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # no __pycache__ in the tree for the modules imported from here on

METRIC = "similarity+MAP eval Gpairs/s at 1/2/4/8 B200 (roofline frac); MAP parity"
UNIT = "Gpairs/s"
BASE_N = 100_000
DIM = 1024
FALLBACK_PEAKS = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}
DUMP_LIMIT_BYTES = 64 * 1024 * 1024


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        with open(path) as f:
            p = json.load(f)
        p["_source"] = "measured"
        return p
    p = dict(FALLBACK_PEAKS)
    p["_source"] = "fallback"
    return p


def load_synth():
    """The synthetic-input generator, loaded by path: importing it through the `wealy_b200` package would load
    libwealy_b200.so, which the reference arm must never touch."""
    path = os.path.join(ROOT, "audio-based-lyrics-matching_b200", "data", "synth.py")
    spec = importlib.util.spec_from_file_location("_wealy_synth", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def workload_config(n_total, world, tracks_override):
    """`config` of the JSON line -- identical for the GPU arm and the reference arm of the same command."""
    if tracks_override:
        what = f"--tracks {n_total} (BASELINE.json configs[2] when 500000)"
    else:
        what = ("BASELINE.json configs[1]" if world == 1 else
                "BASELINE.json configs[1] grown for weak scaling: N_total = 100000*sqrt(n_gpus)")
    return {
        "workload": f"all-vs-all cosine similarity + self/clique mask + rank + AP/MAP/MR1, {n_total} x {DIM} fp32 "
                    f"embeddings, SHS100K-TEST clique-size bootstrap ({what})",
        "tracks": n_total, "dim": DIM, "pairs_per_step": float(n_total) * float(n_total), "n_gpus": world,
    }


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU every 20 ms while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._halt = threading.Event()
        self.ok = False

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {
                "hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4),
                "hw_power_brake": getattr(nv, "nvmlClocksThrottleReasonHwPowerBrakeSlowdown", 0x80),
            }
            self.ok = True
            while not self._halt.is_set():
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                    for k, bit in names.items():
                        if mask & bit:
                            self.reasons.add(k)
                except Exception:
                    pass
                self._halt.wait(0.02)
        except Exception:
            self.ok = False

    def finish(self):
        self._halt.set()
        self.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def dump_outputs(out_dir, per_query, totals, query_rows=None):
    """Writes `per_query` (name -> [n] tensor) and `totals` (name -> small tensor) to out_dir/<name>.npy, float64 tensors
    as float64 and the rest as float32.  `query_rows` (the workload's row of each of the n queries, default 0 .. n-1) goes
    to query_index.npy when given.  Past DUMP_LIMIT_BYTES the per-query arrays keep the same fixed, seeded sample of
    queries, and query_index.npy says which."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    as_np = lambda t: (t.double() if t.dtype == torch.float64 else t.float()).cpu().numpy()
    arrays = {k: as_np(v) for k, v in per_query.items()}
    n = len(next(iter(arrays.values())))
    rows = None if query_rows is None else np.asarray(query_rows, dtype=np.float64)
    keep = min(n, (DUMP_LIMIT_BYTES - 64 * 1024) // (sum(a.itemsize for a in arrays.values()) + 8))
    if keep < n:
        pick = np.sort(torch.randperm(n, generator=torch.Generator().manual_seed(0))[:keep].numpy())
        arrays = {k: a[pick] for k, a in arrays.items()}
        rows = (np.arange(n, dtype=np.float64) if rows is None else rows)[pick]
    if rows is not None:
        arrays["query_index"] = rows
    arrays.update({k: as_np(v) for k, v in totals.items()})
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def physical_gpu_index(local_rank):
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except Exception:
            return local_rank
    return local_rank


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference's own CPU path, bounded sample
# ------------------------------------------------------------------------------------------------
def reference_modules():
    """(tensor_ops, losses) of the UNMODIFIED reference installed under baseline/_ref by baseline/install_ref.py, or
    (None, None): then the CPU legs time the oracle port (kind "port")."""
    try:
        from baseline import install_ref
        mods = install_ref.load()
        return mods if mods else (None, None)
    except Exception:
        return None, None


def cpu_kind(ref_tops):
    if ref_tops is not None:
        return "reference", ("the unmodified reference's lib/tensor_ops.py pairwise_distance_matrix (baseline/_ref) + "
                             "per-query argsort AP/R1 of oracle/evaluator.py (the reference has no evaluator of its own)")
    return "port", "oracle port: torch CPU matmul cosine similarity + per-query argsort AP/R1 (oracle/evaluator.py)"


def run_reference_arm(args):
    import torch
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import evaluator as oev
    synth = load_synth()
    ref_tops, _ = reference_modules()
    dist_fn = ref_tops.pairwise_distance_matrix if ref_tops is not None else None
    kind, how = cpu_kind(ref_tops)
    world = args.gpus
    n_total = int(args.tracks) if args.tracks else int(round(BASE_N * (world ** 0.5)))
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    s = synth.make_eval_set(n_total, DIM, seed=0, md5_ids=False)
    sample = args.cpu_queries
    times = []
    for it in range(args.warmup + args.steps):
        lo = (it * sample) % max(1, n_total - sample)
        t0 = time.perf_counter()
        aps, r1s = oev.evaluate_argsort(s["c"][lo:lo + sample], s["i"][lo:lo + sample], s["z"][lo:lo + sample],
                                        s["c"], s["i"], s["z"], dist_fn=dist_fn)[:2]
        dt = time.perf_counter() - t0
        if it >= args.warmup:
            times.append(dt)
    if args.dump_outputs:   # this arm scores a window of queries per step: the last step's window, with its rows
        dump_outputs(args.dump_outputs, {"aps": aps, "r1s": r1s}, {}, query_rows=range(lo, lo + aps.numel()))
    sec = sum(times) / len(times)
    value = sample * n_total / sec / 1e9
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(n_total, world, args.tracks),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": torch.get_num_threads(), "kind": kind,
                         "sample": f"each step: {sample} queries x {n_total} candidates (bounded sample of the workload); {how}"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# parity of a finished plan against the CPU oracle on a query sample
# ------------------------------------------------------------------------------------------------
def parity_sample(plan, aps, r1s, z_c, c_c, i_c, qsel, *, topk=None, topk_idx=None, topk_sim=None, timed=False):
    """GPU results vs the oracle for the queries `qsel` (CPU index tensor) against the full corpus.
    -> (dict, seconds of the oracle's evaluate_argsort)."""
    import torch
    from oracle import evaluator as oev
    ref_tops, _ = reference_modules()
    t0 = time.perf_counter()
    res_o = oev.evaluate_argsort(c_c[qsel], i_c[qsel], z_c[qsel], c_c, i_c, z_c, topk=topk,
                                 dist_fn=ref_tops.pairwise_distance_matrix if ref_tops is not None else None)
    sec = time.perf_counter() - t0
    aps_o, r1_o = res_o[0], res_o[1]
    qd = qsel.to(aps.device)
    aps_g, r1_g = aps[qd].double().cpu(), r1s[qd].double().cpu()
    out = {"sample_queries": int(qsel.numel()),
           "abs_dMAP": abs(float(aps_g.mean()) - float(aps_o.mean())),
           "rel_dMR1": abs(float(r1_g.mean()) - float(r1_o.mean())) / max(1.0, float(r1_o.mean())),
           "max_abs_dAP": float((aps_g - aps_o).abs().max())}
    # ranks of EVERY relevant item: inside the band its 1e-5 neighbours allow, exact where the band is one rank.  The
    # bands come from the float64 evaluation of the same formula (the arbiter between two fp32-accumulating
    # implementations), on at most 128 of the sampled queries
    qb = qsel[:128]
    off_g, ranks_g, sims_g = (t.cpu() for t in plan.ranks())
    zd = z_c.double()
    off_o, sims_o, exact, lo, hi = oev.rank_bands(c_c[qb], i_c[qb], zd[qb], c_c, i_c, zd, gap=1e-5)
    del zd
    pos = torch.cat([torch.arange(int(off_g[q]), int(off_g[q + 1])) for q in qb.tolist()])
    r, sg = ranks_g[pos].long(), sims_g[pos].double()
    single = lo == hi
    out.update({"item_ranks_queries": int(qb.numel()), "item_ranks_checked": int(r.numel()),
                "item_ranks_out_of_band": int(((r < lo) | (r > hi)).sum()),
                "item_ranks_exact_where_gap_gt_1e-5": int(single.sum()),
                "item_ranks_exact_mismatches": int((r[single] != exact[single]).sum()),
                "max_abs_dsim_relevant_vs_float64": float((sg - sims_o).abs().max()),
                "note": "max_abs_dAP > 0 comes from ranks that moved INSIDE their band (candidates within 1e-5 of a "
                        "relevant item); out_of_band and exact_mismatches must be 0"})
    if topk:
        idx_o, sim_o = res_o[2], res_o[3]
        idx_g, sim_g = topk_idx[qd].cpu(), topk_sim[qd].cpu()
        ok = torch.ones_like(idx_o, dtype=torch.bool)
        ok[:, 1:] &= (sim_o[:, :-1] - sim_o[:, 1:]) > 1e-5
        ok[:, :-1] &= (sim_o[:, :-1] - sim_o[:, 1:]) > 1e-5
        ok[:, -1] = False   # the last position also depends on the (k+1)-th best, which the lists do not show
        out.update({"topk": int(topk), "topk_max_abs_dsim": float((sim_g - sim_o).abs().max()),
                    "topk_idx_compared_where_gap_gt_1e-5": int(ok.sum()),
                    "topk_idx_mismatches": int((idx_g[ok] != idx_o[ok]).sum())})
    return out, sec


def stage_roofline(plan, n, d, passes, total_pairs, peaks, topk=0, parts=4, cap=0):
    """Achieved HBM GB/s of the stages around the sweep (CUDA events inside wealy_eval_run), against the measured
    copy bandwidth.  Algorithmic bytes per stage: DESIGN.md section 4."""
    ms = plan.stage_ms()
    d_pad = -(-d // 64) * 64
    planes = 2 if passes == 3 else 1
    by = {
        "prep": n * d * 4 + n * d_pad * 2 * planes + n * 12,
        "kpos": total_pairs * 2 * d_pad * 2 * planes / 2 + total_pairs * 12,   # every unordered relevant pair's two rows, once
        "ap_reduce": total_pairs * 4 + n * 8,
    }
    if topk:
        # rectangle sweep: 4 streaming lists of `cap` entries per query; symmetric sweep (cap = 0): ~3k + 8 sigma entries
        by["topk_finalize"] = n * (parts * cap if cap else 7 * topk) * 8 + n * topk * 12
    hbm = float(peaks["hbm_gbs"])
    out = {}
    for k, b in by.items():
        t = ms.get(k, 0.0)
        gbs = b / (t * 1e-3) / 1e9 if t > 0 else None
        out[k] = {"ms": t, "bytes": float(b), "gbs": gbs, "frac_of_hbm_peak": (gbs / hbm) if gbs else None}
    out["sweep_ms"] = ms["sweep"]
    out["note"] = ("with top-k in the symmetric sweep the kpos window also holds the sampled pre-pass (one fp16 pass of every query "
                   "against ~N/8 candidates); kpos gathers operand rows of relevant pairs out of L2 (the planes were just written by prep), so its "
                   "'GB/s' is L2-side; ap_reduce / topk_finalize move KB..MB and are launch-latency bound")
    return out


# ------------------------------------------------------------------------------------------------
# extra legs: the other BASELINE.json configs
# ------------------------------------------------------------------------------------------------
def timed_steps(fn, warmup, steps, dev, sync_all):
    import torch
    for _ in range(warmup):
        fn()
    sync_all()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        out = fn()
    e1.record()
    sync_all()
    return e0.elapsed_time(e1) / steps, out


def leg_c1(dev, peaks, precision):
    """configs[0]: SHS100K-TEST-shaped, the case the reference runs on CPU: FULL CPU run beside the GPU."""
    import torch
    from wealy_b200 import evaluation as we
    from wealy_b200.data import synth
    n = 10547
    s = synth.make_eval_set(n, DIM, seed=0)
    c, i, z = s["c"].to(dev), s["i"].to(dev), s["z"].to(dev)
    plan = we.EvalPlan(c, i, c, i, device=dev)
    ms, res = timed_steps(lambda: plan.run(z, z, precision=precision), 3, 10, dev, lambda: torch.cuda.synchronize(dev))
    par, sec = parity_sample(plan, res["aps"], res["r1s"], s["z"], s["c"], s["i"], torch.arange(n))
    plan.close()
    return {"workload": f"{n} x {DIM} all-vs-all, exact SHS100K-TEST clique multiset (1692 cliques)",
            "ms_per_step": ms, "gpairs_per_s": n * n / (ms * 1e-3) / 1e9,
            "cpu_full_run_s": sec, "cpu_gpairs_per_s": n * n / sec / 1e9, "cpu_cores": torch.get_num_threads(),
            "parity_all_queries": par}


def leg_c3(dev, world, rank, peaks, precision, sync_all):
    """configs[2]: 500 000 x 1024 all-vs-all over the N GPUs of this run (strong scaling: total work fixed)."""
    import torch
    import torch.distributed as dist
    from wealy_b200 import evaluation as we, dist as wd
    from wealy_b200.data import synth
    n = 500_000
    s = synth.make_eval_set(n, DIM, seed=3, device=dev, md5_ids=False)
    c, i, z = s["c"], s["i"], s["z"]
    plan = we.EvalPlan(c, i, c, i, device=dev)

    def step():
        if world == 1:
            return plan.run(z, z, precision=precision)
        wd.sharded_step(plan, z, rank, world, precision=precision)
        return plan.finish()

    ms, res = timed_steps(step, 1, 3, dev, sync_all)
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    sweep_ms = plan.last_sweep_ms()
    out = None
    if rank == 0:
        qs = torch.randperm(n, generator=torch.Generator().manual_seed(23))[:64]
        par, _ = parity_sample(plan, res["aps"], res["r1s"], z.cpu(), c.cpu(), i.cpu(), qs)
        peak = float(peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"]))
        tf = 2.0 * n * n / world * DIM / (sweep_ms * 1e-3) / 1e12
        sm = res["sums"].cpu()
        out = {"workload": f"{n} x {DIM} all-vs-all (Discogs-VI full scale), {world} GPU(s), row blocks of the symmetric "
                           f"sweep dealt round-robin, corpus replicated, one all-reduce of the rank counters",
               "scaling": "strong", "n_gpus": world, "ms_per_step": ms, "gpairs_per_s": float(n) * n / (ms * 1e-3) / 1e9,
               "sweep_ms_rank0": sweep_ms, "sweep_algorithmic_tflops_per_gpu": tf, "roofline_frac": tf / peak,
               "map": float(sm[0] / sm[2]), "mr1": float(sm[1] / sm[2]), "parity": par}
    plan.close()
    del s, c, i, z
    torch.cuda.empty_cache()
    return out


def leg_c4(dev, peaks):
    """configs[3]: contrastive loss forward / backward, batch 4096 x 1024 bf16, 4 items per clique."""
    import torch
    from wealy_b200 import losses as wl
    from wealy_b200.data import synth
    from oracle import losses as ol
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import loss_bench as lb
    b, d = 4096, 1024
    s = synth.make_loss_batch(b, d, seed=0, dtype=torch.bfloat16, device=dev)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    peak = float(peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"]))
    out = {"workload": f"NT-Xent / CLEWS forward + backward, batch {b} x {d} bf16, 4 items per clique, L2 flushed between "
                       f"iterations; bf16 inputs take one fp16 tensor-core pass (their 8 significant bits are fewer than it keeps)",
           "algorithmic_flops_fwd_bwd": 8.0 * b * b * d}
    zc = s["z"].float().cpu()
    lab_c, idx_c = s["label"].cpu(), s["idx"].cpu()
    torch.set_num_threads(os.cpu_count() or 1)
    _, ref_losses = reference_modules()
    if ref_losses is not None:      # the unmodified reference modules (baseline/_ref) on the host cores
        out["cpu_kind"] = "reference (lib/losses.py NTXentLoss / CLEWSLoss, fp32, all host cores)"
        ntx_ref, clews_ref = ref_losses.NTXentLoss(0.1), ref_losses.CLEWSLoss()
        cpu_fns = {"ntxent": lambda z: ntx_ref(lab_c.clone(), idx_c, z)[0], "clews": lambda z: clews_ref(lab_c.clone(), idx_c, z)[0]}
    else:
        out["cpu_kind"] = "port (oracle/losses.py, fp32, all host cores)"
        cpu_fns = {"ntxent": lambda z: ol.ntxent(lab_c.clone(), idx_c, z, 0.1)[0], "clews": lambda z: ol.clews(lab_c.clone(), idx_c, z)[0]}
    # (loss_dtype = fp32: the unrounded value; by default the modules round the loss to z's dtype like the reference)
    for name, mod in (("ntxent", wl.NTXentLoss(0.1, loss_dtype=torch.float32)), ("clews", wl.CLEWSLoss(loss_dtype=torch.float32))):
        fn = cpu_fns[name]
        f, lv = lb.gpu_time(mod, s, 20, False, flush)
        fb, _ = lb.gpu_time(mod, s, 20, True, flush)
        rec = {"fwd_ms": f, "fwd_bwd_eager_ms": fb, "loss": lv}
        try:
            gms, glv, ggrad = lb.graph_time(mod, s, 20, flush)
            rec.update({"fwd_bwd_graph_ms": gms, "tflops_graph": 8.0 * b * b * d / (gms * 1e-3) / 1e12,
                        "frac_graph": 8.0 * b * b * d / (gms * 1e-3) / 1e12 / peak})
        except Exception as e:  # report, do not hide
            rec.update({"fwd_bwd_graph_ms": None, "graph_error": repr(e)[:200]})
            ggrad = None
        rec["tflops_eager"] = 8.0 * b * b * d / (fb * 1e-3) / 1e12
        rec["frac_eager"] = rec["tflops_eager"] / peak
        best_f = best_fb = 1e9
        for _ in range(3):
            zz = zc.clone().requires_grad_(True)
            t0 = time.perf_counter(); lo = fn(zz); t1 = time.perf_counter(); lo.backward(); t2 = time.perf_counter()
            best_f, best_fb = min(best_f, t1 - t0), min(best_fb, t2 - t0)
        rec.update({"cpu_fwd_ms": best_f * 1e3, "cpu_fwd_bwd_ms": best_fb * 1e3, "cpu_cores": torch.get_num_threads(),
                    "loss_rel_err_vs_cpu_fp32": abs(lv - float(lo)) / abs(float(lo))})
        if ggrad is not None:
            rec["grad_rel_l2_vs_cpu_fp32"] = float((ggrad.float().cpu() - zz.grad).norm() / zz.grad.norm())
        out[name] = rec
    del flush
    torch.cuda.empty_cache()
    return out


def leg_c5(dev, peaks, precision):
    """configs[4]: lyric-covers multimodal retrieval (text + audio concatenated, 2048-d), ~50k tracks, top-100."""
    import torch
    from wealy_b200 import evaluation as we
    from wealy_b200.data import synth
    n, d, k = 50_000, 2048, 100
    s = synth.make_eval_set(n, d, seed=5, dist="lyric_covers_test", device=dev, md5_ids=False)
    c, i, z = s["c"], s["i"], s["z"]
    plan = we.EvalPlan(c, i, c, i, device=dev)
    ms, res = timed_steps(lambda: plan.run(z, z, topk=k, precision=precision), 3, 5, dev, lambda: torch.cuda.synchronize(dev))
    st = plan.stage_ms()
    qs = torch.randperm(n, generator=torch.Generator().manual_seed(17))[:256]
    par, sec = parity_sample(plan, res["aps"], res["r1s"], z.cpu(), c.cpu(), i.cpu(), qs, topk=k,
                             topk_idx=res["topk_idx"], topk_sim=res["topk_sim"])
    peak = float(peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"]))
    tf = 2.0 * n * n * d / (st["sweep"] * 1e-3) / 1e12
    passes = 3 if precision == "fp16x3" else 1
    out = {"workload": f"{n} x {d} all-vs-all, top-{k} output + AP/R1, lyric-covers-test clique-size bootstrap",
           "ms_per_step": ms, "gpairs_per_s": float(n) * n / (ms * 1e-3) / 1e9,
           "sweep_ms": st["sweep"], "sweep_algorithmic_tflops": tf, "roofline_frac": tf / peak,
           "ceiling_gpairs_per_s_at_d2048": peak * 1e12 / (2.0 * d) / 1e9,
           "topk_path": {1: "symmetric sweep, sampled per-query bounds (csrc/topk_sym_kernels.cuh)", 2: "rectangle sweep, streaming top-k",
                         3: "symmetric sweep overflowed -> rectangle sweep"}.get(plan.last_topk_path(), "?"),
           "stages": stage_roofline(plan, n, d, passes, plan.total_pairs, peaks, topk=k, parts=4,
                                    cap=0 if plan.last_topk_path() == 1 else 320),
           "cpu_sample_gpairs_per_s": 256 * n / sec / 1e9, "cpu_cores": torch.get_num_threads(),
           "parity": par}
    plan.close()
    del s, c, i, z
    torch.cuda.empty_cache()
    return out


def leg_f1(dev, peaks, precision):
    """SURVEY.md 8(f) row f1: chunked tracks all-vs-all (WEALY's test mode: several chunk embeddings per track), the
    chunk distances reduced like distance_tensor_redux(dist, "min") inside the sweep: 12 500 tracks x 8 chunks x 1024."""
    import torch
    from oracle import evaluator as oev
    from wealy_b200 import evaluation as we
    from wealy_b200.data import synth
    n, ch, d = 12_500, 8, DIM
    base = synth.make_eval_set(n, d, seed=8, device=dev, md5_ids=False)
    g = torch.Generator(device=dev).manual_seed(108)
    z = (base["z"][:, None, :] + 0.8 * base["z"].norm(dim=1).mean() / d ** 0.5 * torch.randn(n, ch, d, generator=g, device=dev)).contiguous()
    c, i = base["c"], base["i"]
    plan = we.EvalPlan(c, i, c, i, device=dev)
    sync = lambda: torch.cuda.synchronize(dev)
    out = {"workload": f"{n} tracks x {ch} chunks x {d} all-vs-all, redux=min, chunk embeddings = track embedding + noise"}
    os.environ["WEALY_SYM_TRACKS"] = "0"
    ms_r, res_r = timed_steps(lambda: plan.run(z, z, redux="min", precision=precision, allow_empty=True), 2, 4, dev, sync)
    os.environ.pop("WEALY_SYM_TRACKS")
    ms, res = timed_steps(lambda: plan.run(z, z, redux="min", precision=precision, allow_empty=True), 2, 5, dev, sync)
    sweep = plan.last_sweep_ms()
    stages = plan.stage_ms()
    rows = n * ch
    peak = float(peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"]))
    tf = 2.0 * rows * rows * d / (sweep * 1e-3) / 1e12
    out.update({"ms_per_step": ms, "sweep_ms": sweep, "g_chunk_pairs_per_s": float(rows) * rows / (ms * 1e-3) / 1e9,
                "sweep_algorithmic_tflops": tf, "roofline_frac": tf / peak,
                "path": "half sweep: tiles above the diagonal, every track pair scored for its row and its column query",
                "stages_ms": {k: stages[k] for k in ("prep", "kpos", "sweep", "ap_reduce")},
                "full_rectangle_ms_per_step": ms_r,
                "rectangle_vs_half_identical": bool(torch.equal(res["aps"], res_r["aps"]) and torch.equal(res["r1s"], res_r["r1s"]))})
    # parity: every relevant item's rank of 64 sampled query tracks against the oracle (restated distance_tensor_redux)
    qs = torch.randperm(n, generator=torch.Generator().manual_seed(19))[:64]
    off_g, ranks_g, sims_g = (t.cpu() for t in plan.ranks())
    cc, ic, zc = c.cpu(), i.cpu(), z.cpu()
    t0 = time.perf_counter()
    off_o, sims_o, exact, lo, hi = oev.rank_bands(cc[qs], ic[qs], zc[qs], cc, ic, zc, gap=1e-5, redux="min")
    sec = time.perf_counter() - t0
    pos = torch.cat([torch.arange(int(off_g[q]), int(off_g[q + 1])) for q in qs.tolist()])
    r, sg = ranks_g[pos].long(), sims_g[pos].double()
    single = lo == hi
    out["parity"] = {"sample_query_tracks": int(qs.numel()), "item_ranks_checked": int(r.numel()),
                     "item_ranks_out_of_band": int(((r < lo) | (r > hi)).sum()),
                     "item_ranks_exact_where_gap_gt_1e-5": int(single.sum()),
                     "item_ranks_exact_mismatches": int((r[single] != exact[single]).sum()),
                     "max_abs_dsim_relevant": float((sg - sims_o).abs().max())}
    out["cpu_sample_g_chunk_pairs_per_s"] = 64 * ch * float(rows) / sec / 1e9
    out["cpu_cores"] = torch.get_num_threads()
    plan.close()
    del base, z, c, i
    torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def run_gpu_arm(args):
    import torch
    import torch.distributed as dist
    from wealy_b200 import evaluation as we, dist as wd
    from wealy_b200.data import synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if args.gpus > 1 and world == 1:
        raise SystemExit("launch multi-GPU runs with torch.distributed.run (one process per GPU)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    legs = set(args.legs.split(","))
    torch.set_num_threads(os.cpu_count() or 1)

    n_total = int(args.tracks) if args.tracks else int(round(BASE_N * (world ** 0.5)))
    lo, hi = wd.shard_range(n_total, rank, world)
    s = synth.make_eval_set(n_total, DIM, seed=0, device=dev, md5_ids=False, **({"sigma": args.sigma} if args.sigma else {}))
    z, c, i = s["z"], s["c"], s["i"]
    nq = n_total if world == 1 else (hi - lo)          # queries whose row blocks this rank sweeps (about)
    pairs_total = float(n_total) * float(n_total)

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    # ---- value: inputs resident in HBM, plan built once
    plan = we.EvalPlan(c, i, c, i, device=dev)

    def step_resident():
        if world == 1:
            return plan.run(z, z, precision=args.precision)
        wd.sharded_step(plan, z, rank, world, precision=args.precision)   # two all-reduces: thresholds, rank counters
        return plan.finish()

    for _ in range(args.warmup):
        step_resident()
    sync_all()
    sampler = ClockSampler(physical_gpu_index(local_rank))
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        res = step_resident()
    e1.record()
    sync_all()
    clocks = sampler.finish()
    ms_total = e0.elapsed_time(e1)
    last_sweep_ms = plan.last_sweep_ms()
    t = torch.tensor([ms_total], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item()) / args.steps
    value = pairs_total / (ms_step * 1e-3) / 1e9
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"aps": res["aps"], "r1s": res["r1s"]}, {"sums": res["sums"]})
    s_host = res["sums"].double().cpu()
    gpu_map, gpu_mr1 = float(s_host[0] / s_host[2]), float(s_host[1] / s_host[2])
    passes = 3 if args.precision == "fp16x3" else 1
    peaks = load_peaks()
    stages = stage_roofline(plan, n_total, DIM, passes, plan.total_pairs, peaks) if rank == 0 else None

    # ---- parity at every N: rank 0 scores a query sample with the CPU oracle (also the cpu_baseline sample at N = 1)
    parity = cpu = None
    if rank == 0 and not args.no_cpu:
        nqs = args.cpu_queries if world == 1 else min(args.cpu_queries, 256)
        qs = torch.arange(nqs) if world == 1 else torch.randperm(n_total, generator=torch.Generator().manual_seed(7))[:nqs]
        parity, sec = parity_sample(plan, res["aps"], res["r1s"], z.cpu(), c.cpu(), i.cpu(), qs)
        if world == 1:
            kind, how = cpu_kind(reference_modules()[0])
            cpu = {"value": nqs * n_total / sec / 1e9, "unit": UNIT, "cores": torch.get_num_threads(), "kind": kind,
                   "sample": f"first {nqs} queries x {n_total} candidates in {sec:.1f} s; {how}"}
    sync_all()

    # ---- e2e: public API with HOST pinned buffers, copies + plan build + result read every step
    z_h, c_h, i_h = z.cpu().pin_memory(), c.cpu().pin_memory(), i.cpu().pin_memory()
    # per rank: its 1/world slice of the embeddings (replicated afterwards by one NVLink all-gather) + all ids
    h2d = -(-n_total // world) * DIM * 4 + c_h.numel() * 8 + i_h.numel() * 8
    aps_h = torch.empty(n_total, dtype=torch.float32).pin_memory()
    r1s_h = torch.empty(n_total, dtype=torch.float32).pin_memory()
    d2h = 2 * n_total * 4

    def step_e2e():
        # public API, host tensors in, host tensors out: upload, id plan, evaluation, read-back every step
        if world == 1:
            aps, r1s = we.evaluate(c_h, i_h, z_h, c_h, i_h, z_h, precision=args.precision)
        else:
            out = wd.evaluate_all_vs_all(c_h, i_h, z_h, precision=args.precision)
            aps, r1s = out["aps"], out["r1s"]
        aps_h.copy_(aps, non_blocking=True)
        r1s_h.copy_(r1s, non_blocking=True)
        torch.cuda.current_stream(dev).synchronize()
        if world > 1:
            out["plan"].close()

    def timed_e2e(run_steps):
        sync_all()
        t0 = time.perf_counter()
        e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e2.record()
        run_steps()
        e3.record()
        sync_all()
        wall_ms = (time.perf_counter() - t0) * 1e3
        t = torch.tensor([max(e2.elapsed_time(e3), wall_ms)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    e2e_steps = args.steps
    step_e2e()
    step_e2e()
    single_ms = timed_e2e(lambda: [step_e2e() for _ in range(e2e_steps)]) / e2e_steps
    # `e2e` is the synchronous call at every N (comparable along the scaling series); the double-buffered serving form of the
    # same public API is reported next to it at N = 1 (`e2e.pipelined`)
    e2e_ms, e2e_api = single_ms, ("wealy_b200.evaluation.evaluate" if world == 1 else "wealy_b200.dist.evaluate_all_vs_all") + \
        " (host pinned tensors in, host out; one synchronous call per step: upload, id plan, evaluation, read-back)"
    e2e_route, copy_ms = None, None
    if world == 1:
        # which way the embeddings went in: "host_stream" = wealy_eval_run_host (the device reads the pinned rows itself, in
        # sorted order, while the sweep runs over the rows that have arrived; the same bytes cross PCIe inside the call);
        # the copy-then-compute route (copy engine, then the resident path) is timed beside it
        e2e_route = we.last_path()
        if e2e_route == "host_stream":
            os.environ["WEALY_HOST_STREAM"] = "0"
            try:
                step_e2e()
                copy_ms = timed_e2e(lambda: [step_e2e() for _ in range(e2e_steps)]) / e2e_steps
            finally:
                del os.environ["WEALY_HOST_STREAM"]
            step_e2e()     # (leave the host buffers holding the default route's output)
    if world == 1:
        # the serving form: requests submitted back to back, the upload of request k + 1 on the copy engine while the
        # sweep of request k runs.  Every request still uploads its ids and embeddings, builds its id plan, evaluates and
        # reads its per-query results back -- all inside the timed region.
        pipe = we.EvalPipeline(precision=args.precision)
        pipe.result(pipe.submit(c_h, i_h, z_h))
        last = {}

        def run_pipelined():
            prev = None
            for _ in range(e2e_steps):
                t = pipe.submit(c_h, i_h, z_h)
                if prev is not None:
                    pipe.result(prev)
                prev = t
            a, r = pipe.result(prev)
            last["aps"] = a.clone()
        # warm-up in the same back-to-back pattern: the first requests of a pipeline allocate its slot buffers and grow the
        # library's device pool to two plans alive at once (tens to hundreds of ms each, once per process)
        run_pipelined()
        run_pipelined()
        pipe_ms = timed_e2e(run_pipelined) / e2e_steps
        pipe_dmap = abs(float(last["aps"].double().mean()) - float(aps_h.double().mean()))
        pipe.close()
        pipelined = {"ms_per_step": pipe_ms, "value": pairs_total / (pipe_ms * 1e-3) / 1e9, "unit": UNIT,
                     "abs_dMAP_vs_single_call": pipe_dmap,
                     "api": "wealy_b200.evaluation.EvalPipeline.submit / .result: requests back to back, every request pays its own "
                            "upload (ids + embeddings), id plan, evaluation and read-back inside the timed region; the upload of "
                            "request k+1 runs on the copy engine while the sweep of request k runs"}
    else:
        pipelined = None
    e2e_value = pairs_total / (e2e_ms * 1e-3) / 1e9
    e2e_parity = None
    if rank == 0 and parity is not None:
        # the end-to-end path's own output (host buffers), same sample
        a = aps_h[qs].double()
        e2e_parity = {"abs_dMAP_vs_resident_path": abs(float(a.mean()) - float(res["aps"][qs.to(dev)].double().mean().cpu()))}
    plan.close()
    del z_h, s
    torch.cuda.empty_cache()

    # ---- the other BASELINE configs
    extra = {}
    if "c3" in legs and not args.tracks:
        r = leg_c3(dev, world, rank, peaks, args.precision, sync_all)
        if r is not None:
            extra["c3_500k"] = r
    if world == 1:
        if "c1" in legs:
            extra["c1_shs100k"] = leg_c1(dev, peaks, args.precision)
        if "c4" in legs:
            extra["c4_loss"] = leg_c4(dev, peaks)
        if "c5" in legs:
            extra["c5_topk100"] = leg_c5(dev, peaks, args.precision)
        if "f1" in legs:
            extra["f1_chunked"] = leg_f1(dev, peaks, args.precision)

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (fused sweep), measured live with CUDA events on its stream
    # algorithmic work of this rank's launch: its share of the N_total^2 pairs, 2*D flop each (SURVEY.md 8(d))
    algo_flops = 2.0 * (float(n_total) * n_total / world) * DIM
    achieved = algo_flops / (last_sweep_ms * 1e-3) / 1e12
    # tensor-core work actually issued: the symmetric sweep contracts only the 128 x 256 tiles that reach above
    # the diagonal (row block rb needs column tiles >= rb / 2), times the passes of the precision mode
    n_rb, n_ct = -(-n_total // 128), -(-n_total // 256)
    tiles = sum(max(0, n_ct - rb // 2) for rb in range(rank, n_rb, world))
    executed = 2.0 * 128 * 256 * DIM * tiles * passes / (last_sweep_ms * 1e-3) / 1e12
    peak = float(peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"]))
    variant = "pair" if os.environ.get("WEALY_SYM_PAIR", "1") != "0" else "single"
    # (the capture must be of exactly this kernel: the pair kernel's template carries its number of dense threshold levels)
    variant_key = f"pair_lv{os.environ.get('WEALY_SYM_LEVELS', '4')}" if variant == "pair" else "single"
    traffic, traffic_note = None, "no ncu capture of this exact configuration is committed"
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.isfile(tpath) and world == 1 and not args.tracks:
        try:
            rec = json.load(open(tpath)).get(f"{n_total}x{DIM}_{args.precision}_{variant_key}_1gpu")
            if rec:
                traffic, traffic_note = rec["dram_bytes_per_launch"], f"dram__bytes_read.sum + dram__bytes_write.sum, {rec['source']}"
        except Exception:
            pass
    roofline = {
        "kernel": ("gemm_pair_kernel<EvalSymEpi> (symmetric tcgen05 cta_group::2 similarity sweep over clique-sorted rows + mask + "
                   "rank-count epilogue)" if variant == "pair" else
                   "gemm_kernel<EvalSymEpi> (symmetric tcgen05 similarity sweep over clique-sorted rows + mask + rank-count epilogue)"),
        "bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
        "traffic": traffic, "traffic_note": traffic_note,
        "peak_kind": f"{peaks['_source']} dense bf16/fp16 cuBLAS, sustained (kernel timed inside a long step); "
                     f"burst = {peaks['bf16_tflops']}",
        "frac_of_burst": achieved / float(peaks["bf16_tflops"]),
        "kernel_ms": last_sweep_ms,
        "executed_tflops": executed,
        "frac_executed": executed / peak,
        "stages": stages,
        "note": "achieved = algorithmic flops (2*D per scored pair, both directions of the symmetric sweep) / "
                "kernel time; executed_tflops = tensor-core work issued: half the tiles (symmetry) x 3 passes in "
                "the fp16x3 parity mode (hi*hi + hi*lo + lo*hi)",
    }

    cfg = workload_config(n_total, world, args.tracks)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f16 tensor-core hi/lo split x3, f32 accumulate" if passes == 3 else "f16 tensor-core, f32 accumulate",
        "data": "synthetic",
        "config": cfg,
        "run": {
            "queries_per_gpu": nq,
            "parallelism": ("single GPU" if world == 1 else
                            f"row blocks of the symmetric sweep dealt round-robin to {world} ranks, corpus replicated, "
                            f"one NCCL all-reduce of the int32 rank counters per step"),
            "precision": args.precision, "sweep_kernel": variant,
            "l2": "operand planes %.0f MB per step >> 126 MB L2 (no flush needed)" % (n_total * DIM * 2 * (2 if passes == 3 else 1) / 1e6),
            "map": gpu_map, "mr1": gpu_mr1,
        },
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "ms_per_step": e2e_ms, "api": e2e_api, "route": e2e_route,
                "route_note": None if e2e_route != "host_stream" else (
                    "wealy_eval_run_host: the h2d bytes are read from the pinned buffers by an upload kernel on 8 SMs (rows gathered "
                    "in the plan's sorted order, from the end) INSIDE the timed call, while the symmetric sweep runs over the rows "
                    "that have arrived; results bit-identical to the copy-then-compute route timed beside it"),
                "copy_then_compute": None if copy_ms is None else {
                    "ms_per_step": copy_ms, "value": pairs_total / (copy_ms * 1e-3) / 1e9, "unit": UNIT,
                    "note": "the same call with WEALY_HOST_STREAM=0: cudaMemcpyAsync of the embeddings on a side stream, then the resident path"},
                "pipelined": pipelined},
        "gpu_launches": 5 * args.steps,   # prep, pos_pairs, pos_sort, fused sweep, ap_reduce per step
        "roofline": roofline,
    }
    if e2e_parity:
        line["e2e"].update(e2e_parity)
    if cpu is not None:
        line["cpu_baseline"] = cpu
    if parity is not None:
        line["parity"] = parity
    line.update(extra)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def positive_int(text):
    v = int(text)
    if v < 1:
        raise argparse.ArgumentTypeError(f"must be at least 1, got {v}")
    return v


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=5,
                    help="timed steps of the headline workload and of each of its end-to-end forms; the extra legs "
                         "(c1, c3, c4, c5, f1) time fixed step counts of their own")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--tracks", type=int, default=0,
                    help="override the corpus size of the headline leg; default: 100000 * sqrt(gpus)")
    ap.add_argument("--precision", default=os.environ.get("WEALY_PRECISION", "fp16x3"), choices=["fp16x3", "fp16"])
    ap.add_argument("--cpu-queries", type=int, default=512, help="queries in the bounded CPU sample")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline / parity legs")
    ap.add_argument("--sigma", type=float, default=0.0,
                    help="within-clique noise of the synthetic embeddings (default 2.4: MAP ~0.67; larger = harder data, "
                         "more candidates above the relevant items; diagnostic only)")
    ap.add_argument("--legs", default="main,c1,c3,c4,c5,f1",
                    help="which BASELINE configs to run besides the headline (c1, c3, c4, c5); 'main' = headline only")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step to DIR/<name>.npy (at most 64 MB in all)")
    args = ap.parse_args()
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
