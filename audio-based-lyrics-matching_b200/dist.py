"""Multi-GPU evaluation (SURVEY.md 8(e)): one process per GPU, torch.distributed (NCCL over NVLink / NVSwitch on
the GPU box; gloo in the CPU tests of the merge logic).

Two schemes:

* all-vs-all (queries ARE the corpus, the headline case) -- `evaluate_all_vs_all`: every rank holds the whole
  corpus and sweeps the row blocks rb = rank (mod world) of the SAME symmetric problem (only tiles above the
  diagonal, each element scoring its row and its column query).  A rank therefore holds partial rank counts for
  ALL queries; the one real exchange step of the path is an all-reduce (SUM) of those int32 counters -- the
  "rank counts merged over NCCL" of the north star -- after which every rank owns the complete AP / R1.  Chunked
  tracks ([N, s, D], SURVEY.md 8(f) row f1) shard the chunked sweep the same way for min / max / mean.  Top-k lists
  (per-query state, not counters) are finalized locally, exchanged with one all-to-all so that rank r holds every
  rank's lists of its query slice, merged there and all-gathered.
* general queries vs corpus -- `evaluate_sharded`: queries are independent units, so rank r scores the contiguous
  query slice shard_range(Nq, r, world) against the whole (replicated) corpus with the single-GPU fused kernel and
  the data path needs no collective.  The only exchange is the result merge: one all-reduce of {sum AP, sum R1,
  count} (24 bytes) for MAP / MR1 and, when per-query values are wanted, one all-gather of [Nq/world] x {ap, r1}
  (and of the top-k lists).

Errors are raised on EVERY rank or on none: whatever one rank finds wrong with its share (a query without relevant
candidates) is agreed on with a tiny all-reduce before any rank enters a data collective.
"""
import torch
import torch.distributed as dist


def shard_range(n, rank, world):
    """Contiguous, balanced partition of range(n): the first n % world ranks get one extra item."""
    base, extra = divmod(n, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def merge_sums(local_sums, group=None):
    """All-reduce {sum AP, sum R1, count} -> (MAP, MR1, count) identical on every rank."""
    s = local_sums.detach().clone().double()
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(s, op=dist.ReduceOp.SUM, group=group)
    s = s.cpu()
    n = max(float(s[2]), 1.0)
    return float(s[0]) / n, float(s[1]) / n, int(s[2])


def gather_rows(local, n_total, group=None):
    """All-gather row-sharded results (shard_range layout) into the full [n_total, ...] tensor."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return local
    world = dist.get_world_size(group)
    sizes = [shard_range(n_total, r, world) for r in range(world)]
    longest = max(hi - lo for lo, hi in sizes)
    # (gloo has no all_gather of CUDA tensors: results are staged through the host there -- CPU tests, and two
    #  processes sharing one GPU)
    via_host = local.is_cuda and dist.get_backend(group) == "gloo"
    src = local.cpu() if via_host else local
    pad = torch.zeros((longest,) + tuple(src.shape[1:]), dtype=src.dtype, device=src.device)
    pad[: src.shape[0]] = src
    bufs = [torch.empty_like(pad) for _ in range(world)]
    dist.all_gather(bufs, pad, group=group)
    full = torch.cat([b[: hi - lo] for b, (lo, hi) in zip(bufs, sizes)], dim=0)
    return full.to(local.device) if via_host else full


def upload_sharded(z_host, device, group=None):
    """Host embeddings -> the full [n, d] matrix (or [n, s, d] chunked tracks) on every rank's device without every rank
    pulling the whole corpus over PCIe: rank r uploads only its contiguous 1/world slice of the rows (whole tracks;
    pinned host memory -> HBM), then ONE all-gather over NVLink / NVSwitch replicates the corpus.  Host traffic per rank
    drops from n*d to n*d/world bytes (8 ranks x 1.16 GB through one host bridge at 282k x 1024 was 2/3 of the
    end-to-end step)."""
    on = dist.is_available() and dist.is_initialized()
    world = dist.get_world_size(group) if on else 1
    rank = dist.get_rank(group) if on else 0
    n, row = z_host.shape[0], tuple(z_host.shape[1:])
    if world == 1:
        return z_host.to(device, non_blocking=True)
    chunk = -(-n // world)
    lo, hi = min(rank * chunk, n), min((rank + 1) * chunk, n)
    mine = torch.zeros((chunk,) + row, dtype=z_host.dtype, device=device) if hi - lo < chunk else \
        torch.empty((chunk,) + row, dtype=z_host.dtype, device=device)
    if hi > lo:
        mine[: hi - lo].copy_(z_host[lo:hi], non_blocking=True)
    full = torch.empty((world * chunk,) + row, dtype=z_host.dtype, device=device)
    try:
        dist.all_gather_into_tensor(full, mine, group=group)
    except (RuntimeError, NotImplementedError):      # backends without the flat variant (CPU tests)
        dist.all_gather(list(full.view((world, chunk) + row).unbind(0)), mine, group=group)
    return full[:n]


def exchange_topk(val, idx, cnt, group=None):
    """Every rank's local top-k lists of ALL queries (val [n, k] float32, idx [n, k] int32, cnt [n] int32, as
    EvalPlan.sweep_shard_topk returns them) -> the lists of every rank for THIS rank's query slice
    shard_range(n, rank, world): (val [world, n_r, k], idx [world, n_r, k], cnt [world, n_r]), list w from rank w.
    The rows are already laid out by destination (slices are contiguous), so one all_to_all_single of the three arrays
    packed side by side ([n, 2 k + 1] int32) moves them; gloo stages through the host, as gather_rows does."""
    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    n, k = val.shape
    sizes = [hi - lo for lo, hi in (shard_range(n, r, world) for r in range(world))]
    packed = torch.cat([val.view(torch.int32), idx, cnt[:, None]], dim=1)
    via_host = packed.is_cuda and dist.get_backend(group) == "gloo"
    src = packed.cpu() if via_host else packed
    recv = torch.empty((world * sizes[rank], 2 * k + 1), dtype=torch.int32, device=src.device)
    dist.all_to_all_single(recv, src, output_split_sizes=[sizes[rank]] * world, input_split_sizes=sizes, group=group)
    recv = recv.to(val.device).view(world, sizes[rank], 2 * k + 1)
    return (recv[..., :k].contiguous().view(torch.float32), recv[..., k:2 * k].contiguous(),
            recv[..., 2 * k].contiguous())


def _sym_sharded_topk(plan, z, rank, world, k, *, eps, precision, group):
    """All-vs-all top-k on the row-block-sharded symmetric sweep: every rank sweeps its row blocks with the top-k
    epilogue (sampled bounds computed identically on every rank), the rank counters are summed, the local lists of every
    query slice are exchanged (exchange_topk) and merged on the slice's rank, the merged slices all-gathered.
    -> (dict(aps, r1s, sums, topk_idx, topk_sim), "sym_sharded"); (None, "query_sharded") where the call is not eligible
    (the same on every rank: the decision reads only arguments and ids), (None, "query_sharded_fallback") where some
    rank's merge found a list that overflowed or ended short of k."""
    from .evaluation import merge_topk
    try:
        loc = plan.sweep_shard_topk(z, rank, world, k, eps=eps, precision=precision)
    except NotImplementedError:
        return None, "query_sharded"
    dist.all_reduce(plan.counts_tensor(), op=dist.ReduceOp.SUM, group=group)
    tk_idx, tk_sim, failed = merge_topk(*exchange_topk(loc["val"], loc["idx"], loc["cnt"], group))
    if _agree(failed, plan.device, group):
        return None, "query_sharded_fallback"
    res = plan.finish()
    res["topk_idx"] = gather_rows(tk_idx, plan.nq, group)
    res["topk_sim"] = gather_rows(tk_sim, plan.nq, group)
    return res, "sym_sharded"


def _agree(flag, device, group=None):
    """MAX of a small non-negative integer over the ranks: every rank learns whether ANY rank wants to raise."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return int(flag)
    t = torch.tensor([int(flag)], dtype=torch.int64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
    return int(t.item())


STAGED_MIN_WORLD = 4


def _chunks_per_track(z, chunks, redux, q_chunks):
    """Chunks per track of `z` ([N, s, D], or [N * s, D] with chunks=s; 1 for plain [N, D] embeddings).  Every rank
    passes the same arguments, so whatever this refuses is refused on every rank, before any collective."""
    from . import _native as N
    shape = tuple(torch.as_tensor(z).shape)
    s = shape[1] if len(shape) == 3 else (1 if chunks is None else int(chunks))
    if len(shape) == 3 and chunks is not None and int(chunks) != s:
        raise ValueError(f"chunks={chunks}, but z holds {s} chunks per track")
    if s not in (1, 2, 4, 8, 16):
        raise NotImplementedError("chunks per track must be 1, 2, 4, 8 or 16")
    if redux not in N.REDUX:
        raise NotImplementedError(f"redux {redux!r} is not fused into the evaluation (min / max / mean / meanmin / minmean)")
    if q_chunks is not None and s == 1:
        raise ValueError("chunk counts need chunked tracks")
    return s


def query_slice(queries_z, q_chunks, lo, hi, chunks=None):
    """Query tracks [lo, hi) of `queries_z` ([N, D], [N, s, D], or [N * s, D] with chunks=s) and their chunk counts."""
    s = 1 if (queries_z.ndim == 3 or chunks is None) else int(chunks)
    return queries_z[lo * s:hi * s], None if q_chunks is None else torch.as_tensor(q_chunks)[lo:hi]


def sharded_step(plan, z, rank, world, *, eps=1e-6, precision=None, group=None, redux="min", q_chunks=None, chunks=None):
    """The multi-GPU all-vs-all sweep up to (not including) finish(): the relevant similarities are computed once across
    the ranks (each rank its share of the queries; one all-reduce of floats assembles them -- every element has a single
    non-zero contribution, so the sum is exact), every rank sweeps the row blocks rank (mod world) of the symmetric
    problem, and the per-(query, relevant item) rank counters are summed (the second all-reduce).  Chunked tracks
    (`chunks`, `redux`, `q_chunks` as in EvalPlan.run) take the row-block-sharded chunked sweep the same way."""
    kw = dict(eps=eps, precision=precision, redux=redux, q_chunks=q_chunks, chunks=chunks)
    if world >= STAGED_MIN_WORLD:
        plan.shard_prepare(z, rank, world, **kw)
        dist.all_reduce(plan.thresholds_tensor(), op=dist.ReduceOp.SUM, group=group)
        plan.shard_sweep(rank, world)
    else:
        # two or three ranks: recomputing the relevant similarities on every rank (0.5 ms at 141k tracks) costs less
        # than the extra collective (measured at N = 2: 23.1 vs 23.5 ms per step)
        plan.sweep_shard(z, rank, world, **kw)
    dist.all_reduce(plan.counts_tensor(), op=dist.ReduceOp.SUM, group=group)


def evaluate_all_vs_all(c, i, z, *, precision=None, eps=1e-6, group=None, plan=None, allow_empty=False, topk=None,
                        chunks=None, redux="min", q_chunks=None):
    """All-vs-all evaluation of one set (clique ids c, version ids i, embeddings z) over all ranks of `group`.
    Every rank passes the full tensors (host embeddings are uploaded 1/world per rank and all-gathered over
    NVLink).  -> dict(map, mr1, count, aps, r1s, plan); identical on every rank.

    Chunked tracks (SURVEY.md 8(f) row f1): z [N, s, D] (or [N * s, D] with chunks=s), `redux` and ragged `q_chunks`
    as in EvalPlan.run.  min / max / mean shard the chunked sweep by row blocks, like plain embeddings; meanmin /
    minmean (d(q, c) != d(c, q), so no half sweep) take the query-partitioned scheme below.

    topk -> also topk_idx / topk_sim and, with more than one rank, topk_path.  Top-k lists are per-query state, not
    additive counters: where the single-GPU run takes the symmetric top-k sweep (plain [N, D] embeddings, k <= 128,
    N >= max(16384, 192 k)) and world * k <= 1024, every rank sweeps its row blocks with the top-k epilogue, the rank
    counters are summed, each rank merges every rank's lists of its query slice (one all-to-all) and the merged slices
    are all-gathered (topk_path "sym_sharded").  Otherwise -- and, on every rank, when a merge finds a list that
    overflowed or ended short of k ("query_sharded_fallback") -- the query-partitioned scheme (`evaluate_sharded`:
    every rank scores its slice of the queries against the replicated corpus with the streaming top-k, the lists are
    all-gathered; "query_sharded").

    Like EvalPlan.run, a query without any relevant candidate raises ValueError unless allow_empty -- on every
    rank (all ranks build the same id plan), before the first collective."""
    from .evaluation import EvalPlan
    on = dist.is_available() and dist.is_initialized()
    rank = dist.get_rank(group) if on else 0
    world = dist.get_world_size(group) if on else 1
    s = _chunks_per_track(z, chunks, redux, q_chunks)
    if world > 1 and s > 1 and (topk or redux in ("meanmin", "minmean")):
        if not torch.as_tensor(z).is_cuda:
            z = upload_sharded(torch.as_tensor(z), torch.device("cuda", torch.cuda.current_device()), group)
        out = evaluate_sharded(c, i, z, c, i, z, topk=topk, precision=precision, eps=eps, group=group,
                               allow_empty=allow_empty, chunks=chunks, redux=redux, q_chunks=q_chunks, c_chunks=q_chunks)
        if topk:
            out["topk_path"] = "query_sharded"
        return out
    side = None
    if world > 1 and not torch.as_tensor(z).is_cuda:
        # 1/world of the rows per rank + NVLink all-gather, issued on a side stream BEFORE the id plan is built: the
        # copy engine and NCCL move the embeddings while the plan's small kernels and host read-backs run
        device = plan.device if plan is not None else torch.device("cuda", torch.cuda.current_device())
        from .evaluation import side_stream
        side = side_stream(device)
        side.wait_stream(torch.cuda.current_stream(device))
        with torch.cuda.stream(side):
            z = upload_sharded(torch.as_tensor(z), device, group)
    own = plan is None
    if own:
        plan = EvalPlan(c, i, c, i)
    if side is not None:
        torch.cuda.current_stream(plan.device).wait_stream(side)
        z.record_stream(torch.cuda.current_stream(plan.device))
    if plan.queries_without_relevant and not allow_empty:
        raise ValueError(f"{plan.queries_without_relevant} queries have no relevant candidate "
                         "(every clique needs >= 2 versions; pass allow_empty=True to score the rest)")
    if world == 1:
        res = plan.run(z, z, eps=eps, precision=precision, allow_empty=allow_empty, topk=topk, chunks=chunks, redux=redux,
                       q_chunks=q_chunks)
    elif topk:
        res, path = _sym_sharded_topk(plan, z, rank, world, min(int(topk), plan.nq), eps=eps, precision=precision,
                                      group=group)
        if res is None:
            if own:
                plan.close()
            out = evaluate_sharded(c, i, z, c, i, z, topk=topk, precision=precision, eps=eps, group=group,
                                   allow_empty=allow_empty)
            out["topk_path"] = path
            return out
    else:
        sharded_step(plan, z, rank, world, eps=eps, precision=precision, group=group, redux=redux, q_chunks=q_chunks,
                     chunks=chunks)
        res = plan.finish()
    s = res["sums"].cpu()                                            # one 24-byte device -> host read
    n = max(float(s[2]), 1.0)
    out = {"map": float(s[0]) / n, "mr1": float(s[1]) / n, "count": int(s[2]), "aps": res["aps"], "r1s": res["r1s"],
           "plan": plan}
    if topk and "topk_idx" in res:
        out["topk_idx"], out["topk_sim"] = res["topk_idx"], res["topk_sim"]
    if topk and world > 1:
        out["topk_path"] = path
    return out


def evaluate_sharded(queries_c, queries_i, queries_z, candidates_c, candidates_i, candidates_z, *, topk=None,
                     precision=None, eps=1e-6, gather=True, group=None, plan=None, allow_empty=False, chunks=None,
                     redux="min", q_chunks=None, c_chunks=None):
    """Every rank passes the FULL query / candidate tensors (or its own copy of them); rank r
    scores its slice.  Returns dict(map, mr1, count[, aps, r1s, topk_idx, topk_sim]) on every rank.

    Chunked tracks: `chunks`, `redux` and the ragged `q_chunks` / `c_chunks` as in EvalPlan.run; rank r passes the chunk
    counts of its query slice, `c_chunks` whole.

    A rank whose slice is empty (world > Nq) contributes nothing; a query without relevant candidates raises
    ValueError on EVERY rank (agreed on before the merge collectives) unless allow_empty."""
    from .evaluation import EvalPlan
    on = dist.is_available() and dist.is_initialized()
    rank = dist.get_rank(group) if on else 0
    world = dist.get_world_size(group) if on else 1
    _chunks_per_track(queries_z, chunks, redux, q_chunks if q_chunks is not None else c_chunks)
    if (q_chunks is None) != (c_chunks is None):
        if queries_z is not candidates_z:
            raise ValueError("q_chunks and c_chunks go together")
        q_chunks = c_chunks = q_chunks if c_chunks is None else c_chunks
    nq = len(queries_c)
    lo, hi = shard_range(nq, rank, world)
    device = plan.device if plan is not None else torch.device("cuda", torch.cuda.current_device())
    own = plan is None
    if own and hi > lo:
        plan = EvalPlan(queries_c[lo:hi], queries_i[lo:hi], candidates_c, candidates_i, device=device)
    bad = 0 if plan is None else int(plan.queries_without_relevant)
    bad = _agree(bad if not allow_empty else 0, device, group)
    if bad:
        raise ValueError("some queries have no relevant candidate (every clique needs >= 2 versions; "
                         "pass allow_empty=True to score the rest)")
    k = 0 if topk is None else min(int(topk), len(candidates_c))
    if hi > lo:
        qz, ql = query_slice(queries_z, q_chunks, lo, hi, chunks)
        res = plan.run(qz, candidates_z, topk=topk, eps=eps, precision=precision, allow_empty=allow_empty, chunks=chunks,
                       redux=redux, q_chunks=ql, c_chunks=c_chunks)
    else:                                                            # empty shard: neutral contribution
        res = {"aps": torch.empty(0, dtype=torch.float32, device=device),
               "r1s": torch.empty(0, dtype=torch.float32, device=device),
               "sums": torch.zeros(3, dtype=torch.float64, device=device)}
        if k:
            res["topk_idx"] = torch.empty((0, k), dtype=torch.long, device=device)
            res["topk_sim"] = torch.empty((0, k), dtype=torch.float32, device=device)
    m, r1, cnt = merge_sums(res["sums"], group)
    out = {"map": m, "mr1": r1, "count": cnt, "plan": plan}
    if gather:
        out["aps"] = gather_rows(res["aps"], nq, group)
        out["r1s"] = gather_rows(res["r1s"], nq, group)
        if topk:
            out["topk_idx"] = gather_rows(res["topk_idx"], nq, group)
            out["topk_sim"] = gather_rows(res["topk_sim"], nq, group)
    return out
