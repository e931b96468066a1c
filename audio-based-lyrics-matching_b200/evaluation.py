"""Retrieval evaluation on sm_100a: self / same-clique masking by id, per-query ranking,
AP / MAP / MR1 and optional top-k, fused into the similarity sweep (wealy_eval_run).

The reference has not released its evaluator (SURVEY.md 8(a7)); the interface is inferred from the
evaluation tensors it prepares (`candidates_c`, `candidates_i`: lib/audio_dataset/dataset.py:82-86,
448-449), positives / self follow lib/losses.py:40-42 and the distance is
`pairwise_distance_matrix(q, cands, mode="cos")` (lib/tensor_ops.py:167-173):

    aps, r1s = evaluate(queries_c, queries_i, queries_z, candidates_c, candidates_i, candidates_z)
    aps, r1s, topk_idx, topk_sim = evaluate(..., topk=100)

Host tensors are accepted and copied to the current CUDA device (that copy is part of the
end-to-end measurement in bench.py); the computation itself has no CPU path.  float64 embeddings are
rounded to float32 on entry: the outputs are ranks, AP / R1 and float32 top-k similarities, and the rounding
moves a similarity by < 2e-7, far inside the 1e-5 gap below which ranks are allowed to differ.
"""
import ctypes

import torch

from . import _native as N
from .tensor_ops import passes_of


def _to_device(t, device, dtype=None):
    t = torch.as_tensor(t)
    if dtype is not None and t.dtype != dtype:
        t = t.to(dtype)
    if not t.is_cuda:
        t = t.to(device, non_blocking=True)
    return t


class EvalPlan:
    """Everything that depends on ids only (clique-sorted candidate order, per-query relevant
    segments, CSR offsets) -- build once per (queries, candidates) id set, run for any embeddings."""

    def __init__(self, queries_c, queries_i, candidates_c, candidates_i, device=None, host_z=None, eps=1e-6, precision=None):
        """host_z (optional): the pinned host embeddings run_host() will be called with (same eps / precision) -- their
        upload then starts inside the plan build, as soon as the sorted order exists (wealy_eval_plan_create_host)."""
        if device is None:
            device = torch.device("cuda", torch.cuda.current_device())
        self.device = torch.device(device)
        same = (queries_c is candidates_c) and (queries_i is candidates_i)
        self.q_c = _to_device(queries_c, self.device, torch.long).contiguous().view(-1)
        self.q_i = _to_device(queries_i, self.device, torch.long).contiguous().view(-1)
        if same:
            self.c_c, self.c_i = self.q_c, self.q_i
        else:
            self.c_c = _to_device(candidates_c, self.device, torch.long).contiguous().view(-1)
            self.c_i = _to_device(candidates_i, self.device, torch.long).contiguous().view(-1)
        assert self.q_c.numel() == self.q_i.numel() and self.c_c.numel() == self.c_i.numel()
        self.nq, self.nc = self.q_c.numel(), self.c_c.numel()
        self._handle = ctypes.c_void_p()
        with torch.cuda.device(self.device):
            if host_z is not None and host_z.ndim == 2 and host_z.stride(1) == 1:
                N.check(N.lib.wealy_eval_plan_create_host(
                    self.q_c.data_ptr(), self.q_i.data_ptr(), self.nq, self.c_c.data_ptr(), self.c_i.data_ptr(), self.nc,
                    host_z.data_ptr(), host_z.stride(0), host_z.shape[1], N.dtype_code(host_z.dtype), float(eps),
                    passes_of(precision), N.stream_ptr(self.device), ctypes.byref(self._handle)))
                self._keepalive = host_z
            else:
                N.check(N.lib.wealy_eval_plan_create(
                    self.q_c.data_ptr(), self.q_i.data_ptr(), self.nq, self.c_c.data_ptr(), self.c_i.data_ptr(), self.nc,
                    N.stream_ptr(self.device), ctypes.byref(self._handle)))
        tp, nr, mr = ctypes.c_int64(), ctypes.c_int64(), ctypes.c_int64()
        N.check(N.lib.wealy_eval_plan_info(self._handle, ctypes.byref(tp), ctypes.byref(nr), ctypes.byref(mr)))
        self.total_pairs, self.queries_without_relevant, self.max_relevant = tp.value, nr.value, mr.value

    def close(self):
        if getattr(self, "_handle", None) is not None and self._handle.value:
            N.lib.wealy_eval_plan_destroy(self._handle)
            self._handle = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- multi-GPU all-vs-all: symmetric sweep sharded by row blocks, rank counts summed over ranks ----
    def _shard_input(self, z, chunks, redux, q_chunks):
        """-> (z [rows, D] on the device, chunks per track, device int32 chunk counts or None) for the sharded entries;
        chunked tracks come as [N, s, D] or as [N * s, D] with chunks=s, as in run()."""
        z = _to_device(z, self.device)
        if z.dtype == torch.float64:
            z = z.float()
        if z.ndim == 3:
            assert chunks is None or int(chunks) == z.shape[1]
            chunks = z.shape[1]
            z = z.reshape(-1, z.shape[-1])
        s = 1 if chunks is None else int(chunks)
        if s not in (1, 2, 4, 8, 16):
            raise NotImplementedError("chunks per track must be 1, 2, 4, 8 or 16")
        if redux not in N.REDUX:
            raise NotImplementedError(f"redux {redux!r} is not fused into the evaluation (min / max / mean / meanmin / minmean)")
        if q_chunks is not None and s == 1:
            raise ValueError("chunk counts need chunked tracks")
        assert z.ndim == 2 and z.shape[0] == self.nq * s and self.nq == self.nc
        if z.stride(1) != 1:
            z = z.contiguous()
        lens = None
        if q_chunks is not None:
            lens = torch.as_tensor(q_chunks).to(self.device, torch.int32).contiguous()
            assert lens.shape == (self.nq,)
        return z, s, lens

    def sweep_shard(self, z, shard_rank, shard_world, *, eps=1e-6, precision=None, redux="min", q_chunks=None, chunks=None):
        """Sweep this rank's share (row blocks = shard_rank mod shard_world) of the symmetric all-vs-all
        problem; the plan must have been built with queries == candidates.  Chunked tracks ([N, s, D], or [N * s, D]
        with chunks=s; `redux`, ragged `q_chunks` as in run()) take the row-block-sharded chunked sweep."""
        z, s, lens = self._shard_input(z, chunks, redux, q_chunks)
        with torch.cuda.device(self.device):
            if s == 1:
                N.check(N.lib.wealy_eval_sweep_shard(
                    self._handle, z.data_ptr(), z.stride(0), z.shape[1], N.dtype_code(z.dtype), float(eps),
                    passes_of(precision), int(shard_rank), int(shard_world), N.stream_ptr(self.device)))
            else:
                N.check(N.lib.wealy_eval_sweep_shard_tracks(
                    self._handle, z.data_ptr(), z.stride(0), z.shape[1], N.dtype_code(z.dtype), float(eps),
                    passes_of(precision), s, N.REDUX[redux], None if lens is None else lens.data_ptr(), int(shard_rank),
                    int(shard_world), N.stream_ptr(self.device)))
        self._keepalive = (z, lens)

    def sweep_shard_topk(self, z, shard_rank, shard_world, k, *, eps=1e-6, precision=None):
        """sweep_shard() with top-k lists: this rank's row blocks of the symmetric top-k sweep (plain [N, D] embeddings;
        the sampled per-query bounds are computed on every rank, identically).  The rank counters stay in the plan (sum
        counts_tensor() over the ranks, then finish()); returns this rank's local lists dict(val [N, k] float32,
        idx [N, k] int32, cnt [N] int32): per query the min(k, m) best of its m local candidates, by descending
        similarity, ties to the lower index, padded with (-inf, -1); cnt = m, or -1 where the list overflowed.  Merge
        the lists of all ranks with merge_topk().  Raises NotImplementedError, before any work and alike on every rank,
        where the single-GPU run would not take the symmetric top-k sweep or shard_world * k > 1024."""
        z, _, _ = self._shard_input(z, None, "min", None)
        k = int(k)
        val = torch.empty((self.nq, max(k, 0)), dtype=torch.float32, device=self.device)
        idx = torch.empty((self.nq, max(k, 0)), dtype=torch.int32, device=self.device)
        cnt = torch.empty(self.nq, dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            N.check(N.lib.wealy_eval_sweep_shard_topk(
                self._handle, z.data_ptr(), z.stride(0), z.shape[1], N.dtype_code(z.dtype), float(eps),
                passes_of(precision), k, int(shard_rank), int(shard_world), val.data_ptr(), idx.data_ptr(), cnt.data_ptr(),
                N.stream_ptr(self.device)))
        self._keepalive = z
        return {"val": val, "idx": idx, "cnt": cnt}

    def shard_prepare(self, z, shard_rank, shard_world, *, eps=1e-6, precision=None, redux="min", q_chunks=None,
                      chunks=None):
        """Stage 1 of the sharded sweep: planes of the whole corpus, thresholds of THIS rank's share of the queries.
        Then sum thresholds_tensor() over the ranks and call shard_sweep() (which reuses this call's layout)."""
        z, s, lens = self._shard_input(z, chunks, redux, q_chunks)
        self._shard_dim, self._shard_passes = z.shape[1], passes_of(precision)
        self._shard_tracks = (s, redux, lens)
        with torch.cuda.device(self.device):
            if s == 1:
                N.check(N.lib.wealy_eval_shard_prepare(
                    self._handle, z.data_ptr(), z.stride(0), z.shape[1], N.dtype_code(z.dtype), float(eps),
                    self._shard_passes, int(shard_rank), int(shard_world), N.stream_ptr(self.device)))
            else:
                N.check(N.lib.wealy_eval_shard_prepare_tracks(
                    self._handle, z.data_ptr(), z.stride(0), z.shape[1], N.dtype_code(z.dtype), float(eps),
                    self._shard_passes, s, N.REDUX[redux], None if lens is None else lens.data_ptr(), int(shard_rank),
                    int(shard_world), N.stream_ptr(self.device)))
        self._keepalive = (z, lens)

    def thresholds_tensor(self):
        """float32 view (no copy) of {lowest thresholds, all thresholds} (after a chunked shard_prepare(): the thresholds
        alone, in the CSR order of ranks()): what a multi-GPU run all-reduces (SUM) between shard_prepare() and
        shard_sweep()."""
        ptr, n = ctypes.c_void_p(), ctypes.c_int64()
        N.check(N.lib.wealy_eval_plan_thresholds(self._handle, ctypes.byref(ptr), ctypes.byref(n)))

        class _Dev:
            __cuda_array_interface__ = {"shape": (n.value,), "typestr": "<f4", "data": (ptr.value, False), "version": 2}
        return torch.as_tensor(_Dev(), device=self.device)

    def shard_sweep(self, shard_rank, shard_world, *, redux=None, q_chunks=None, chunks=None):
        """Stage 2: this rank's row blocks of the symmetric sweep on the planes / thresholds stage 1 left in the plan.
        redux / q_chunks / chunks default to what shard_prepare() was given; a different redux or chunks raises
        ValueError (the thresholds were computed for those)."""
        if not hasattr(self, "_shard_dim"):
            raise AssertionError("shard_sweep() needs shard_prepare() first")
        s, red, lens = self._shard_tracks
        if (chunks is not None and int(chunks) != s) or (redux is not None and redux != red):
            raise ValueError(f"shard_prepare() ran with chunks={s}, redux={red!r}")
        if q_chunks is not None:
            lens = torch.as_tensor(q_chunks).to(self.device, torch.int32).contiguous()
            assert lens.shape == (self.nq,)
            self._shard_tracks = (s, red, lens)
        with torch.cuda.device(self.device):
            if s == 1:
                N.check(N.lib.wealy_eval_shard_sweep(self._handle, self._shard_dim, self._shard_passes, int(shard_rank),
                                                     int(shard_world), N.stream_ptr(self.device)))
            else:
                N.check(N.lib.wealy_eval_shard_sweep_tracks(
                    self._handle, self._shard_dim, self._shard_passes, s, N.REDUX[red],
                    None if lens is None else lens.data_ptr(), int(shard_rank), int(shard_world),
                    N.stream_ptr(self.device)))

    def counts_tensor(self):
        """int32 view (no copy) of the plan's per-(query, relevant item) rank counters: the buffer a
        multi-GPU run all-reduces between sweep_shard() and finish()."""
        ptr, n = ctypes.c_void_p(), ctypes.c_int64()
        N.check(N.lib.wealy_eval_plan_counts(self._handle, ctypes.byref(ptr), ctypes.byref(n)))

        class _Dev:
            __cuda_array_interface__ = {"shape": (n.value,), "typestr": "<i4", "data": (ptr.value, False), "version": 2}
        return torch.as_tensor(_Dev(), device=self.device)

    def finish(self):
        """Rank counts -> dict(aps, r1s, sums) for ALL queries."""
        aps = torch.empty(self.nq, dtype=torch.float32, device=self.device)
        r1s = torch.empty(self.nq, dtype=torch.float32, device=self.device)
        sums = torch.empty(3, dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            N.check(N.lib.wealy_eval_finish(self._handle, aps.data_ptr(), r1s.data_ptr(), sums.data_ptr(),
                                            N.stream_ptr(self.device)))
        return {"aps": aps, "r1s": r1s, "sums": sums}

    def ranks(self):
        """Per-item ranks of the last run: (offsets[nq + 1] int64, ranks[total_pairs] int32, sims[total_pairs] f32);
        query q's relevant candidates, best first, are ranks[offsets[q]:offsets[q + 1]] (1-based rank among all
        non-self candidates) with their cosine similarities."""
        n = max(int(self.total_pairs), 1)
        offsets = torch.empty(self.nq + 1, dtype=torch.long, device=self.device)
        ranks = torch.empty(n, dtype=torch.int32, device=self.device)
        sims = torch.empty(n, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            N.check(N.lib.wealy_eval_plan_ranks(self._handle, offsets.data_ptr(), ranks.data_ptr(), sims.data_ptr(),
                                                N.stream_ptr(self.device)))
        return offsets, ranks[: self.total_pairs], sims[: self.total_pairs]

    def last_sweep_ms(self):
        """Device time of the fused similarity+ranking kernel of the last run (CUDA events)."""
        ms = ctypes.c_float()
        N.check(N.lib.wealy_eval_plan_last_sweep_ms(self._handle, ctypes.byref(ms)))
        return ms.value

    def last_topk_path(self):
        """0 none, 1 symmetric sweep (sampled bounds), 2 rectangle sweep (streaming top-k), 3 symmetric failed -> rectangle."""
        v = ctypes.c_int()
        N.check(N.lib.wealy_eval_plan_last_topk_path(self._handle, ctypes.byref(v)))
        return v.value

    def stage_ms(self):
        """Device time of the stages of the last run: dict(prep, kpos, sweep, ap_reduce, topk_finalize) in ms."""
        ms = (ctypes.c_float * 5)()
        N.check(N.lib.wealy_eval_plan_stage_ms(self._handle, ms))
        return dict(zip(("prep", "kpos", "sweep", "ap_reduce", "topk_finalize"), (float(v) for v in ms)))

    def run_host(self, z, *, eps=1e-6, precision=None, allow_empty=False):
        """All-vs-all evaluation of PINNED HOST embeddings `z[N, D]` -> dict(aps, r1s, sums) on the device: the device
        reads the rows itself, in the plan's sorted order and from the end, while the symmetric sweep already runs over
        what has arrived (wealy_eval_run_host) -- no separate upload.  Raises NotImplementedError where that pipeline
        does not apply (then upload and call run()); `z` must stay alive until the current stream has drained (the plan
        keeps a reference until its next run)."""
        if self.queries_without_relevant and not allow_empty:
            raise ValueError(f"{self.queries_without_relevant} queries have no relevant candidate "
                             "(every clique needs >= 2 versions; pass allow_empty=True to score the rest)")
        assert z.ndim == 2 and z.shape[0] == self.nq == self.nc
        if z.stride(1) != 1:
            raise NotImplementedError("run_host needs contiguous rows")
        aps = torch.empty(self.nq, dtype=torch.float32, device=self.device)
        r1s = torch.empty(self.nq, dtype=torch.float32, device=self.device)
        sums = torch.empty(3, dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            N.check(N.lib.wealy_eval_run_host(
                self._handle, z.data_ptr(), z.stride(0), z.shape[1], N.dtype_code(z.dtype), float(eps),
                passes_of(precision), aps.data_ptr(), r1s.data_ptr(), sums.data_ptr(), N.stream_ptr(self.device)))
        self._keepalive = z
        return {"aps": aps, "r1s": r1s, "sums": sums}

    def run(self, queries_z, candidates_z, *, topk=None, eps=1e-6, precision=None, allow_empty=False, chunks=None,
            redux="min", q_chunks=None, c_chunks=None):
        """-> dict(aps, r1s, sums[, topk_idx, topk_sim]); `sums` = device doubles {sum AP, sum R1, #scored}.

        Chunked tracks (SURVEY.md 8(f) row f1): pass `[N, s, D]` embeddings (or `[N * s, D]` with `chunks=s`,
        s in {2, 4, 8, 16}): the s x s chunk distances of every track pair are reduced like
        `distance_tensor_redux(dist, redux)` (lib/tensor_ops.py:288-373; redux in min / max / mean / meanmin /
        minmean) inside the sweep's epilogue before ranking; ids and results are per track.

        Ragged tracks: `q_chunks[Nq]` / `c_chunks[Nc]` = valid chunks of every track (1 .. s; the remaining rows are
        padding): reduced like `distance_tensor_redux(dist, redux, mask)` with mask = query chunk invalid | candidate
        chunk invalid."""
        if self.queries_without_relevant and not allow_empty:
            raise ValueError(f"{self.queries_without_relevant} queries have no relevant candidate "
                             "(every clique needs >= 2 versions; pass allow_empty=True to score the rest)")
        same = queries_z is candidates_z
        qz = _to_device(queries_z, self.device)
        cz = qz if same else _to_device(candidates_z, self.device)
        if qz.dtype == torch.float64:                     # (see the module docstring)
            qz = qz.float()
            cz = qz if same else cz.float()
        if qz.ndim == 3:                                  # [N, s, D]: the chunks of a track
            assert cz.ndim == 3 and cz.shape[1] == qz.shape[1] and (chunks is None or int(chunks) == qz.shape[1])
            chunks = qz.shape[1]
            qz = qz.reshape(-1, qz.shape[-1])
            cz = qz if same else cz.reshape(-1, cz.shape[-1])
        s = 1 if chunks is None else int(chunks)
        if s not in (1, 2, 4, 8, 16):
            raise NotImplementedError("chunks per track must be 1, 2, 4, 8 or 16")
        if redux not in N.REDUX:
            raise NotImplementedError(f"redux {redux!r} is not fused into the evaluation (min / max / mean / meanmin / minmean)")
        assert qz.ndim == 2 and cz.ndim == 2 and qz.shape[1] == cz.shape[1]
        assert qz.shape[0] == self.nq * s and cz.shape[0] == self.nc * s
        if qz.dtype != cz.dtype:
            raise RuntimeError("queries_z and candidates_z must have the same dtype")
        if qz.stride(1) != 1:
            qz = qz.contiguous()
            cz = qz if same else cz
        if cz.stride(1) != 1:
            cz = cz.contiguous()
        k = 0 if topk is None else min(int(topk), self.nc)
        aps = torch.empty(self.nq, dtype=torch.float32, device=self.device)
        r1s = torch.empty(self.nq, dtype=torch.float32, device=self.device)
        sums = torch.empty(3, dtype=torch.float64, device=self.device)
        tk_idx = torch.empty((self.nq, k), dtype=torch.long, device=self.device) if k else None
        tk_sim = torch.empty((self.nq, k), dtype=torch.float32, device=self.device) if k else None
        if (q_chunks is None) != (c_chunks is None):
            if not same:
                raise ValueError("q_chunks and c_chunks go together")
            q_chunks = c_chunks = q_chunks if c_chunks is None else c_chunks
        if q_chunks is not None:
            if s == 1:
                raise ValueError("chunk counts need chunked tracks")
            ql = torch.as_tensor(q_chunks).to(self.device, torch.int32).contiguous()
            cl = ql if c_chunks is q_chunks else torch.as_tensor(c_chunks).to(self.device, torch.int32).contiguous()
            assert ql.shape == (self.nq,) and cl.shape == (self.nc,)
            with torch.cuda.device(self.device):
                N.check(N.lib.wealy_eval_run_ragged(
                    self._handle, qz.data_ptr(), qz.stride(0), cz.data_ptr(), cz.stride(0), qz.shape[1],
                    N.dtype_code(qz.dtype), float(eps), passes_of(precision), k, s, N.REDUX[redux], ql.data_ptr(),
                    cl.data_ptr(), aps.data_ptr(), r1s.data_ptr(), sums.data_ptr(), tk_idx.data_ptr() if k else None,
                    tk_sim.data_ptr() if k else None, N.stream_ptr(self.device)))
            ql.record_stream(torch.cuda.current_stream(self.device))
            cl.record_stream(torch.cuda.current_stream(self.device))
            out = {"aps": aps, "r1s": r1s, "sums": sums}
            if k:
                out["topk_idx"], out["topk_sim"] = tk_idx, tk_sim
            return out
        with torch.cuda.device(self.device):
            N.check(N.lib.wealy_eval_run_chunked(
                self._handle, qz.data_ptr(), qz.stride(0), cz.data_ptr(), cz.stride(0), qz.shape[1],
                N.dtype_code(qz.dtype), float(eps), passes_of(precision), k, s, N.REDUX[redux], aps.data_ptr(),
                r1s.data_ptr(), sums.data_ptr(), tk_idx.data_ptr() if k else None, tk_sim.data_ptr() if k else None,
                N.stream_ptr(self.device)))
        out = {"aps": aps, "r1s": r1s, "sums": sums}
        if k:
            out["topk_idx"], out["topk_sim"] = tk_idx, tk_sim
        return out


def merge_topk(val, idx, cnt):
    """Merge the local top-k lists of `world` ranks (EvalPlan.sweep_shard_topk), restricted to the same n queries:
    val [world, n, k] float32, idx [world, n, k] int32, cnt [world, n] int32 on one CUDA device ->
    (topk_idx [n, k] int64, topk_sim [n, k] float32, failed): per query the k best of its world * k entries, by
    descending similarity, ties to the lower index, whatever the order of the world lists.  `failed` counts the queries
    whose lists overflowed (cnt -1) or hold fewer than k entries together: their lists are not the k best (recompute
    them).  Synchronises the stream once (to read `failed`).  k <= 128 and world * k <= 1024."""
    assert val.ndim == 3 and idx.shape == val.shape and cnt.shape == val.shape[:2]
    assert val.is_cuda and idx.is_cuda and cnt.is_cuda
    world, n, k = val.shape
    device = val.device
    val = val.to(torch.float32).contiguous()
    idx = idx.to(torch.int32).contiguous()
    cnt = cnt.to(torch.int32).contiguous()
    out_idx = torch.empty((n, k), dtype=torch.long, device=device)
    out_sim = torch.empty((n, k), dtype=torch.float32, device=device)
    fail = torch.zeros(1, dtype=torch.int32, device=device)
    with torch.cuda.device(device):
        N.check(N.lib.wealy_eval_topk_merge(val.data_ptr(), idx.data_ptr(), cnt.data_ptr(), world, n, k,
                                            out_idx.data_ptr(), out_sim.data_ptr(), fail.data_ptr(), N.stream_ptr(device)))
    return out_idx, out_sim, int(fail.item())


def evaluate(queries_c, queries_i, queries_z, candidates_c, candidates_i, candidates_z, *, topk=None, mode="cos",
             eps=1e-6, precision=None, allow_empty=False, plan=None, chunks=None, redux="min", q_chunks=None,
             c_chunks=None):
    """-> (aps[Nq], r1s[Nq]) or (aps, r1s, topk_idx[Nq,k], topk_sim[Nq,k]) on the CUDA device.

    AP_q = 1/P sum_{p relevant} rank_rel(p) / rank_all(p); R1_q = rank of the best relevant item;
    self (candidates_i == queries_i) is excluded, relevant = same clique and not self."""
    if mode not in ("cos", "cossim"):
        raise NotImplementedError("wealy_b200.evaluate ranks by cosine distance (mode='cos')")
    own = plan is None
    # all-vs-all over pinned host embeddings: upload, normalisation and sweep run as one pipeline (EvalPlan.run_host)
    host = (topk is None and chunks is None and q_chunks is None and c_chunks is None
            and _host_streamable(queries_c, queries_i, queries_z, candidates_c, candidates_i, candidates_z))
    if own:
        side = None
        if not host:
            # host embeddings: start their upload on a side stream FIRST, so that the copy engine moves them while the id
            # plan is built (a handful of small kernels and two host read-backs on the current stream)
            queries_z, candidates_z, side = _prefetch_to_device(queries_z, candidates_z)
        plan = EvalPlan(queries_c, queries_i, candidates_c, candidates_i, host_z=queries_z if host else None, eps=eps,
                        precision=precision)
        if side is not None:
            torch.cuda.current_stream(plan.device).wait_stream(side)
            for t in {id(queries_z): queries_z, id(candidates_z): candidates_z}.values():
                t.record_stream(torch.cuda.current_stream(plan.device))
    try:
        res = None
        if host:
            try:
                res = plan.run_host(queries_z, eps=eps, precision=precision, allow_empty=allow_empty)
            except NotImplementedError:     # (e.g. equal shapes but different ids on the two sides): upload and run
                res = None
        _last_path[0] = "host_stream" if res is not None else "device"
        if res is None:
            res = plan.run(queries_z, candidates_z, topk=topk, eps=eps, precision=precision, allow_empty=allow_empty,
                           chunks=chunks, redux=redux, q_chunks=q_chunks, c_chunks=c_chunks)
    finally:
        if own:
            torch.cuda.current_stream(plan.device).synchronize()
            plan.close()
    if topk is None:
        return res["aps"], res["r1s"]
    return res["aps"], res["r1s"], res["topk_idx"], res["topk_sim"]


def _host_streamable(queries_c, queries_i, queries_z, candidates_c, candidates_i, candidates_z):
    """True when evaluate() hands the embeddings to wealy_eval_run_host: one pinned host matrix on both sides, rows of
    4 k <= 1024 contiguous elements, and enough of them for the pipeline to pay (below ~24 k rows the sweep is shorter
    than the upload and the copy engine, which overlaps with the id plan, is the faster way in).
    WEALY_HOST_STREAM=0 keeps the copy-then-compute path, WEALY_HOST_STREAM_MIN_ROWS moves the threshold."""
    import os
    z = queries_z
    if os.environ.get("WEALY_HOST_STREAM", "1") == "0" or not isinstance(z, torch.Tensor):
        return False
    if not (z is candidates_z and queries_c is candidates_c and queries_i is candidates_i):
        return False
    if z.ndim != 2 or z.shape[0] < int(os.environ.get("WEALY_HOST_STREAM_MIN_ROWS", "24576")):
        return False
    return (not z.is_cuda and z.is_pinned() and z.ndim == 2 and z.dtype in (torch.float32, torch.float16, torch.bfloat16)
            and z.stride(1) == 1 and z.stride(0) % 4 == 0 and z.shape[1] % 4 == 0 and 0 < z.shape[1] <= 1024
            and z.data_ptr() % 16 == 0)


_last_path = ["device"]


def last_path():
    """Which route the last evaluate() of this process took: "host_stream" (wealy_eval_run_host) or "device"."""
    return _last_path[0]


_side_streams = {}


def side_stream(device):
    """One upload stream per device, kept for the life of the process: torch's caching allocator hands a block back only
    to the stream it was allocated on, so a fresh stream per call would cudaMalloc the embeddings' buffer every time."""
    device = torch.device(device)
    key = device.index if device.index is not None else torch.cuda.current_device()
    if key not in _side_streams:
        _side_streams[key] = torch.cuda.Stream(device)
    return _side_streams[key]


def _prefetch_to_device(queries_z, candidates_z):
    """Host tensors -> device copies issued on a side stream (pinned memory makes them asynchronous); returns the
    (possibly replaced) tensors and the stream to wait on, or None when nothing had to move."""
    qz, cz = torch.as_tensor(queries_z), torch.as_tensor(candidates_z)
    if qz.is_cuda and cz.is_cuda:
        return queries_z, candidates_z, None
    device = torch.device("cuda", torch.cuda.current_device())
    side = side_stream(device)
    side.wait_stream(torch.cuda.current_stream(device))
    same = queries_z is candidates_z
    with torch.cuda.stream(side):
        qd = qz if qz.is_cuda else qz.to(device, non_blocking=True)
        cd = qd if same else (cz if cz.is_cuda else cz.to(device, non_blocking=True))
    return qd, cd, side


class EvalPipeline:
    """Back-to-back all-vs-all evaluations of HOST-resident sets (serving / periodic evaluation during training): the
    host -> device upload of request k + 1 runs on a copy stream while the sweep of request k occupies the SMs, and the
    per-query results come back through pinned host buffers.  Every request still pays everything itself -- upload of
    ids and embeddings, id plan, evaluation, read-back --; only the copy engine and the SMs work at the same time.

        pipe = EvalPipeline()
        t0 = pipe.submit(c, i, z)                # returns at once (the id plan build synchronises with the previous sweep)
        t1 = pipe.submit(c2, i2, z2)
        aps, r1s = pipe.result(t0)               # pinned host tensors, valid until `depth` more requests have been submitted

    Single process / single GPU; `precision`, `eps` as in evaluate().  The first requests of a pipeline allocate its slot
    buffers and grow the library's device pool to `depth` plans alive at once (tens to hundreds of ms each, once); after
    that a request costs what its upload / sweep cost (C2: 25 ms per request against 29.3 ms for evaluate())."""

    def __init__(self, depth=2, device=None, precision=None, eps=1e-6, allow_empty=False, redux="min"):
        assert depth >= 2
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.depth, self.precision, self.eps, self.allow_empty = int(depth), precision, float(eps), bool(allow_empty)
        self.redux = redux                                        # chunked tracks (z [N, s, D]): see EvalPlan.run
        self.copy_stream = side_stream(self.device)
        self.slots = [dict(z=None, c=None, i=None, aps=None, r1s=None, done=None, plan=None) for _ in range(self.depth)]
        self.count = 0

    def _buffers(self, slot, z, c, i):
        n = z.shape[0]
        if slot["z"] is None or slot["z"].shape != z.shape or slot["z"].dtype != z.dtype:
            with torch.cuda.stream(self.copy_stream):        # (allocated on the stream that fills them)
                slot["z"] = torch.empty(tuple(z.shape), dtype=z.dtype, device=self.device)
                slot["c"] = torch.empty(n, dtype=torch.long, device=self.device)
                slot["i"] = torch.empty(n, dtype=torch.long, device=self.device)
            for t in (slot["z"], slot["c"], slot["i"]):
                t.record_stream(torch.cuda.current_stream(self.device))
            slot["aps"] = torch.empty(n, dtype=torch.float32).pin_memory()
            slot["r1s"] = torch.empty(n, dtype=torch.float32).pin_memory()

    def submit(self, c, i, z):
        """Enqueue one all-vs-all evaluation of host tensors (pin them for an asynchronous upload) -> ticket.
        z: [N, D] embeddings, or [N, s, D] chunked tracks (reduced with the pipeline's `redux`)."""
        z, c, i = torch.as_tensor(z), torch.as_tensor(c).long(), torch.as_tensor(i).long()
        assert z.ndim in (2, 3) and z.shape[0] == c.numel() == i.numel()
        z = z.contiguous()
        if z.dtype == torch.float64:
            z = z.float()
        slot = self.slots[self.count % self.depth]
        if slot["plan"] is not None:                          # the request that used this slot `depth` submits ago
            slot["done"].synchronize()
            slot["plan"].close()
            slot["plan"] = None
        self._buffers(slot, z, c, i)
        compute = torch.cuda.current_stream(self.device)
        with torch.cuda.stream(self.copy_stream):
            slot["z"].copy_(z, non_blocking=True)
            slot["c"].copy_(c, non_blocking=True)
            slot["i"].copy_(i, non_blocking=True)
            uploaded = torch.cuda.Event()
            uploaded.record(self.copy_stream)
        compute.wait_event(uploaded)
        with torch.cuda.device(self.device):
            plan = EvalPlan(slot["c"], slot["i"], slot["c"], slot["i"], device=self.device)
            try:
                res = plan.run(slot["z"], slot["z"], eps=self.eps, precision=self.precision, allow_empty=self.allow_empty,
                               redux=self.redux)
            except Exception:
                plan.close()                                      # (e.g. queries without a relevant candidate: the slot stays free)
                raise
            slot["aps"].copy_(res["aps"], non_blocking=True)
            slot["r1s"].copy_(res["r1s"], non_blocking=True)
            slot["done"] = torch.cuda.Event()
            slot["done"].record(compute)
        # (the next upload into this slot waits for this sweep on the host: see the top of submit())
        slot["plan"], slot["sums"] = plan, res["sums"]
        self.count += 1
        return self.count - 1

    def result(self, ticket):
        """-> (aps, r1s) pinned host tensors of request `ticket` (blocks until its read-back has finished)."""
        if not (self.count - self.depth <= ticket < self.count):
            raise ValueError("the result of this request has been overwritten (more than `depth` requests ago)")
        slot = self.slots[ticket % self.depth]
        slot["done"].synchronize()
        return slot["aps"], slot["r1s"]

    def close(self):
        for slot in self.slots:
            if slot["plan"] is not None:
                slot["done"].synchronize()
                slot["plan"].close()
                slot["plan"] = None


def pool_stats(device=None):
    """Device scratch of the library on `device` (its private stream-ordered pool; torch's allocator is not involved):
    dict(reserved, used, reserved_high, used_high) in bytes."""
    v = [ctypes.c_int64() for _ in range(4)]
    with torch.cuda.device(torch.cuda.current_device() if device is None else device):
        N.check(N.lib.wealy_pool_stats(*[ctypes.byref(x) for x in v]))
    return dict(zip(("reserved", "used", "reserved_high", "used_high"), (x.value for x in v)))


def release_scratch(device=None):
    """Give all idle device scratch of the library back to the driver (synchronises the device); live plans keep theirs."""
    with torch.cuda.device(torch.cuda.current_device() if device is None else device):
        N.check(N.lib.wealy_pool_release())


def mean_metrics(sums):
    """(MAP, MR1) from the device `sums` vector -- one 24-byte device->host read."""
    s = sums.detach().to("cpu")
    n = max(float(s[2]), 1.0)
    return float(s[0]) / n, float(s[1]) / n
