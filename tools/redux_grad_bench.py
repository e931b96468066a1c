"""Forward + backward of distance_tensor_redux and of the masked reductions, timed with CUDA events after warm-up.

Three arms on the same CUDA tensors: the fused autograd Functions (wealy_distance_redux / wealy_masked_reduce and
their backward kernels), the `fused=False` composition of masked reductions (redux only), and the oracle's torch
composition (oracle/masked.py, the reference op for op).  Every working set is far above the 126 MB L2, so no flush is
needed between iterations.  For the one-pass cases the backward's minimal HBM traffic (inputs read once, dx written
once) over its time is reported against 7.7 TB/s; best-k and bpwr are bound by the per-warp selection: time only.
Prints one JSON line (and writes it to --out)."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import wealy_b200  # noqa: E402,F401
from wealy_b200 import tensor_ops as wt  # noqa: E402
from oracle import masked as om  # noqa: E402

HBM_PEAK = 7.7e12
STRATEGIES = ["min", "max", "mean", "minmean", "meanmin", "best-4", "worst-4", "bpwr", "smin", "smeanmin", "sbpwr"]
ONE_PASS = {"min", "max", "mean", "minmean", "meanmin", "smin", "smeanmin"}


def _median_ms(fn, reps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    ms.sort()
    return ms[len(ms) // 2]


def _time_arm(f, x, reps, warmup):
    """(forward + backward ms, backward-only ms) of f at x, upstream gradient of ones."""
    xg = x.detach().requires_grad_(True)
    out = f(xg)
    g = torch.ones_like(out)

    def step():
        xg.grad = None
        f(xg).backward(g)
    fb = _median_ms(step, reps, warmup)
    bw = _median_ms(lambda: torch.autograd.grad(out, xg, g, retain_graph=True), reps, warmup)
    return fb, bw


def _card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, check=True).stdout.strip().splitlines()[0]
        name, power = (s.strip() for s in q.split(","))
    except (OSError, subprocess.CalledProcessError, IndexError, ValueError):
        name, power = torch.cuda.get_device_name(), "unknown"
    return {"gpu": name, "power_limit": power}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--redux-shape", type=int, nargs=4, default=[1024, 1024, 8, 8])
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("redux_grad_bench needs a CUDA device")
    res = {"card": _card(), "reps": a.reps, "warmup": a.warmup, "redux": {}, "masked": {}}
    gen = torch.Generator(device="cuda").manual_seed(0)
    shape = tuple(a.redux_shape)
    dist = torch.rand(shape, device="cuda", generator=gen) * 2
    mask = torch.rand(shape, device="cuda", generator=gen) < 0.2
    n = dist.numel()
    bwd_bytes = n * (4 + 1 + 4) + shape[0] * shape[1] * 4          # dist + mask read, ddist written, g read
    res["redux"]["shape"] = list(shape)
    for r in STRATEGIES:
        row = {}
        for arm, f in (("fused", lambda t: wt.distance_tensor_redux(t, r, mask=mask)),
                       ("composition", lambda t: wt.distance_tensor_redux(t, r, mask=mask, fused=False)),
                       ("oracle", lambda t: om.distance_tensor_redux(t, r, mask=mask))):
            fb, bw = _time_arm(f, dist, a.reps, a.warmup)
            row[arm] = {"fwd_bwd_ms": round(fb, 4), "bwd_ms": round(bw, 4)}
        if r in ONE_PASS:
            gbs = bwd_bytes / (row["fused"]["bwd_ms"] * 1e-3)
            row["fused"]["bwd_min_bytes"] = bwd_bytes
            row["fused"]["bwd_GBps"] = round(gbs / 1e9, 1)
            row["fused"]["bwd_share_of_hbm_peak"] = round(gbs / HBM_PEAK, 3)
        res["redux"][r] = row
        print(r, json.dumps(row), file=sys.stderr)
    for rows, cols in ((4096, 65536), (64, 4194304)):
        x = torch.randn(rows, cols, device="cuda", generator=gen)
        m = torch.rand(rows, cols, device="cuda", generator=gen) < 0.2
        key = f"{rows}x{cols}"
        res["masked"][key] = {}
        for fn in ("mmean", "mmin"):
            row = {}
            for arm, mod in (("fused", wt), ("oracle", om)):
                fb, bw = _time_arm(lambda t: getattr(mod, fn)(t, mask=m, dim=1), x, a.reps, a.warmup)
                row[arm] = {"fwd_bwd_ms": round(fb, 4), "bwd_ms": round(bw, 4)}
            # minimal traffic of the backward: mean reads the mask and writes dx; min also reads x
            nbytes = rows * cols * (1 + 4 + (4 if fn == "mmin" else 0)) + rows * 4
            gbs = nbytes / (row["fused"]["bwd_ms"] * 1e-3)
            row["fused"].update(bwd_min_bytes=nbytes, bwd_GBps=round(gbs / 1e9, 1), bwd_share_of_hbm_peak=round(gbs / HBM_PEAK, 3))
            res["masked"][key][fn] = row
            print(key, fn, json.dumps(row), file=sys.stderr)
        del x, m
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
