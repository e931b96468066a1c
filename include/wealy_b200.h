/* wealy_b200.h -- C ABI of the B200-native (sm_100a) WEALY retrieval-and-scoring hot path.
 *
 * The reference (helemanc/audio-based-lyrics-matching) is pure Python / PyTorch: the path has
 * no FFI of its own, only Python call signatures (SURVEY.md section 8(b)).  This header is the
 * drop-in boundary a binding for that path talks to: plain pointers and sizes, no torch types,
 * every entry point returns an int status (0 = ok) and never throws; wealy_last_error() returns
 * the message of the last failure on the calling thread.  The Python mirror of the reference
 * interface (package `wealy_b200`: tensor_ops / losses / evaluation) binds these symbols with
 * ctypes; INTEGRATION.md shows the stub a maintainer of the reference would add.
 *
 * All data pointers are DEVICE pointers on the current CUDA device unless stated otherwise.
 * `stream` is a cudaStream_t passed as void* (0 = legacy default stream).  Calls are
 * asynchronous with respect to the host unless documented otherwise.
 */
#ifndef WEALY_B200_H_
#define WEALY_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- status codes ---------------------------------------------------------------------- */
#define WEALY_OK 0
#define WEALY_ERR_BAD_ARG 1      /* null pointer, negative size, unknown enum (AssertionError / NotImplementedError upstream) */
#define WEALY_ERR_UNSUPPORTED 2  /* valid in the reference but not built here (e.g. cdist with p != 2) */
#define WEALY_ERR_CUDA 3         /* a CUDA runtime / driver call failed; see wealy_last_error() */
#define WEALY_ERR_WORKSPACE 4    /* workspace too small */
#define WEALY_ERR_ID_RANGE 5     /* a clique / version id does not fit in 32 bits */

/* ---- enums ----------------------------------------------------------------------------- */
/* element type of embedding / output buffers */
#define WEALY_F32 0
#define WEALY_F16 1
#define WEALY_BF16 2
#define WEALY_F64 3 /* accepted by wealy_masked_reduce; matrices of doubles go through wealy_sim_matrix_f64 */

/* pairwise_distance_matrix modes -- lib/tensor_ops.py:157-173 */
#define WEALY_MODE_COSSIM 0
#define WEALY_MODE_COS 1
#define WEALY_MODE_DOTSIM 2
#define WEALY_MODE_DOT 3
#define WEALY_MODE_SQEUC 4  /* also nsqeuc via `post` = 1/D */
#define WEALY_MODE_EUC 5    /* fro/euc with p = 2; nfro/neuc via `post` = D^-1/2 */

/* tensor-core precision of the contraction */
#define WEALY_PASSES_FP16 1   /* one fp16 pass: |err| ~ 1e-4 on unit vectors (fast mode) */
#define WEALY_PASSES_FP16X3 3 /* hi*hi + hi*lo + lo*hi: |err| ~ 1e-6, fp32-grade (parity mode, default) */

const char* wealy_last_error(void);
int wealy_version(void);
/* Device scratch of the library on the CURRENT device: plans and temporaries come from a private stream-ordered pool
 * (nothing is taken from, or returned to, the caller's allocator -- the reference's functions allocate through torch;
 * this is the C ABI's equivalent).  Bytes reserved from the driver / in use now, and their high-water marks.  Destroying
 * a plan releases idle scratch above WEALY_POOL_KEEP_MB (default 4096) back to the driver. */
int wealy_pool_stats(int64_t* reserved_bytes, int64_t* used_bytes, int64_t* reserved_high, int64_t* used_high);
/* Give ALL idle scratch of the current device back to the driver now (synchronises the device). */
int wealy_pool_release(void);

/* ---- a1/a2: materialised similarity / distance matrix ------------------------------------
 * Replaces lib/tensor_ops.py:152-176 `pairwise_distance_matrix(x, y, mode, p, eps)` (modes
 * cos/cossim/dot/dotsim/sqeuc/nsqeuc and the p = 2 cdist modes) and lib/tensor_ops.py:131-149
 * `pairwise_euclidean_distance_matrix`.
 *   x [n, d] (row stride ldx elements), y [m, d] (ldy); out [n, m] (row stride ld_out), out_dtype.
 *   eps: the reference's `eps` added to the L2 norm (cos modes).  post: output scale for the
 *   n* modes.  workspace: wealy_sim_matrix_workspace_bytes(n, m, d, passes) bytes.            */
size_t wealy_sim_matrix_workspace_bytes(int64_t n, int64_t m, int64_t d, int passes);
int wealy_sim_matrix(const void* x, int64_t n, int64_t ldx, const void* y, int64_t m, int64_t ldy, int64_t d,
                     int in_dtype, int mode, float eps, float post, int passes, void* out, int64_t ld_out,
                     int out_dtype, void* workspace, size_t workspace_bytes, void* stream);

/* float64 operands (the reference returns its input dtype): the same modes on a CUDA-core DGEMM, every number a double.
 * workspace: wealy_sim_matrix_f64_workspace_bytes(n, m) bytes.  The evaluation and loss entry points take
 * float32 / float16 / bfloat16 only: their Python mirrors round float64 inputs to float32 (documented there).        */
size_t wealy_sim_matrix_f64_workspace_bytes(int64_t n, int64_t m);
int wealy_sim_matrix_f64(const double* x, int64_t n, int64_t ldx, const double* y, int64_t m, int64_t ldy, int64_t d, int mode,
                         double eps, double post, double* out, int64_t ld_out, void* workspace, size_t workspace_bytes,
                         void* stream);

/* Gradient of the cosine modes of pairwise_distance_matrix (the reference differentiates through it,
 * lib/losses.py:45).  grad [n][m] = dL/d(out) and grad_t [m][n] = its transpose (both with the input dtype);
 * dx [n][d], dy [m][d] receive dL/dx, dL/dy (pass x == y twice and add the two when the operands are the same tensor). */
size_t wealy_sim_matrix_backward_workspace_bytes(int64_t n, int64_t m, int64_t d, int passes);
int wealy_sim_matrix_backward(const void* x, int64_t n, int64_t ldx, const void* y, int64_t m, int64_t ldy, int64_t d,
                              int in_dtype, int mode, float eps, int passes, const void* grad, int64_t ld_grad,
                              const void* grad_t, int64_t ld_grad_t, void* dx, int64_t ld_dx, void* dy, int64_t ld_dy,
                              void* workspace, size_t workspace_bytes, void* stream);

/* Gradient of the dot modes (dot / dotsim): dx [n][d] = G y, dy [m][d] = G^T x.  grad [n][m] and grad_t [m][n] are the
 * upstream gradient and its transpose (negated by the caller for mode "dot" = 1 - x.y), xt [d][n] / yt [d][m] the
 * transposed operands; all with the input dtype.                                                                     */
size_t wealy_dot_matrix_backward_workspace_bytes(int64_t n, int64_t m, int64_t d, int passes);
int wealy_dot_matrix_backward(const void* grad, int64_t ld_grad, const void* grad_t, int64_t ld_grad_t, const void* xt,
                              int64_t ld_xt, const void* yt, int64_t ld_yt, int64_t n, int64_t m, int64_t d, int dtype,
                              int passes, void* dx, int64_t ld_dx, void* dy, int64_t ld_dy, void* workspace,
                              size_t workspace_bytes, void* stream);

/* ---- a7: fused retrieval evaluation -------------------------------------------------------
 * Self / same-clique masking by id, per-query ranking, AP / R1 (and optional top-k) without
 * materialising the Nq x Nc matrix.  The evaluator is not in the reference; argument vocabulary
 * follows lib/audio_dataset/dataset.py:82-86,448-449 (candidates_c / candidates_i), positives
 * and self follow lib/losses.py:40-42, distance follows lib/tensor_ops.py:167-173 mode "cos".
 *
 * A plan holds everything that depends on ids only (clique-sorted candidate order, per-query
 * relevant segments, CSR offsets) plus cached device scratch; create it once per (queries,
 * candidates) id set and run it for any embeddings.  plan_create synchronises the stream
 * (it returns counts to the host); run / destroy do not allocate after the first run.        */
typedef struct wealy_eval_plan wealy_eval_plan;

int wealy_eval_plan_create(const int64_t* queries_c, const int64_t* queries_i, int64_t nq,
                           const int64_t* candidates_c, const int64_t* candidates_i, int64_t nc, void* stream,
                           wealy_eval_plan** plan);
/* host-side facts computed at creation: total (query, same-clique candidate) pairs, number of
 * queries without any relevant candidate, largest number of relevant candidates of a query.  */
int wealy_eval_plan_info(const wealy_eval_plan* plan, int64_t* total_pairs, int64_t* queries_without_relevant,
                         int64_t* max_relevant);
/* queries_z [nq, d] (row stride ld_q), candidates_z [nc, d] (ld_c), same dtype.
 * aps, r1s: [nq] float (NaN for a query without relevant candidates).
 * sums: 3 doubles on the device = {sum AP, sum R1, number of scored queries}  (MAP = sums[0]/sums[2]).
 * topk > 0: topk_idx [nq, topk] int64 (-1 padded), topk_sim [nq, topk] float (-inf padded),
 *           best first, self excluded; pass NULL / 0 to skip.                                 */
int wealy_eval_run(wealy_eval_plan* plan, const void* queries_z, int64_t ld_q, const void* candidates_z, int64_t ld_c,
                   int64_t d, int dtype, float eps, int passes, int topk, float* aps, float* r1s, double* sums,
                   int64_t* topk_idx, float* topk_sim, void* stream);
/* The all-vs-all case (plan built with queries == candidates, no top-k) for embeddings that are still in PINNED HOST
 * memory: host_z [n, d] (row stride ld; d = 4 k <= 1024, 16-byte aligned) is read by the device itself -- a small
 * persistent kernel on a few SMs of its own gathers the caller's rows over PCIe in the plan's clique-sorted order, from
 * the last rows backwards -- while the symmetric sweep already runs over the rows that have arrived: upload,
 * normalisation and sweep as one pipeline instead of copy-then-compute (the caller of the reference would `.cuda()` the
 * embeddings first: lib/losses.py:45 / lib/tensor_ops.py:167-173 take device tensors).  Results are bit-identical to
 * wealy_eval_run on a device copy of host_z.  Work is enqueued on `stream` and on an internal upload stream ordered
 * with it; host_z must stay valid until `stream` has drained.  A device pointer is accepted and takes the plain path;
 * WEALY_ERR_UNSUPPORTED for pageable memory, other shapes or plans (callers then upload and use wealy_eval_run).
 * Environment: WEALY_HOST_UP_SMS (SMs of the upload kernel, default 8; 0 = next to the sweep's CTAs),
 * WEALY_HOST_PARTS (1 / 2 / 5 / 7 parts instead of the size-based choice), WEALY_HOST_TRACE=1 (per-part time stamps
 * on stderr; synchronises).                                                                                    */
int wealy_eval_run_host(wealy_eval_plan* plan, const void* host_z, int64_t ld, int64_t d, int dtype, float eps, int passes,
                        float* aps, float* r1s, double* sums, void* stream);
/* wealy_eval_plan_create for a plan that wealy_eval_run_host will run on host_z (same ld / d / dtype / eps / passes): the
 * upload of the first rows starts as soon as the clique-sorted order exists and proceeds under the rest of the plan
 * build (CSR offsets, collision maps, host read-backs) instead of behind it.  Anything wealy_eval_run_host would refuse
 * (pageable memory, other shapes, queries != candidates) simply creates the plan without the early upload; a run on
 * other embeddings ignores it.                                                                                  */
int wealy_eval_plan_create_host(const int64_t* queries_c, const int64_t* queries_i, int64_t nq,
                                const int64_t* candidates_c, const int64_t* candidates_i, int64_t nc, const void* host_z,
                                int64_t ld, int64_t d, int dtype, float eps, int passes, void* stream,
                                wealy_eval_plan** plan);

/* f1 (SURVEY.md section 8(f)): evaluation of CHUNKED tracks -- every track has `chunks` (1, 2, 4, 8 or 16) embeddings,
 * queries_z [nq * chunks, d] / candidates_z [nc * chunks, d] (the chunks of a track are consecutive rows), the plan's ids
 * are per track.  The chunk-level cosine distances of a track pair are reduced like
 * distance_tensor_redux(dist[b1, b2, s1, s2], redux) of lib/tensor_ops.py:288-373 INSIDE the sweep's epilogue (the 4-D
 * tensor is never materialised), then ranked as in wealy_eval_run.  topk_sim holds 1 - reduced distance.             */
enum { WEALY_REDUX_MIN = 0, WEALY_REDUX_MAX = 1, WEALY_REDUX_MEAN = 2, WEALY_REDUX_MEANMIN = 3, WEALY_REDUX_MINMEAN = 4 };
int wealy_eval_run_chunked(wealy_eval_plan* plan, const void* queries_z, int64_t ld_q, const void* candidates_z,
                           int64_t ld_c, int64_t d, int dtype, float eps, int passes, int topk, int chunks, int redux,
                           float* aps, float* r1s, double* sums, int64_t* topk_idx, float* topk_sim, void* stream);
/* Ragged tracks: as wealy_eval_run_chunked, but track t has only q_len[t] / c_len[t] valid chunks (device int32
 * [nq] / [nc], values 1 .. chunks; the rows of the remaining chunks are padding and may hold anything finite).
 * Padding is excluded exactly like the mask argument of distance_tensor_redux (lib/tensor_ops.py:288-373, mask =
 * query chunk invalid OR candidate chunk invalid; True = excluded, `:186`): min / max over the valid chunk pairs,
 * means divided by the valid counts.                                                                            */
int wealy_eval_run_ragged(wealy_eval_plan* plan, const void* queries_z, int64_t ld_q, const void* candidates_z,
                          int64_t ld_c, int64_t d, int dtype, float eps, int passes, int topk, int chunks, int redux,
                          const int32_t* q_len, const int32_t* c_len, float* aps, float* r1s, double* sums,
                          int64_t* topk_idx, float* topk_sim, void* stream);
/* Multi-GPU all-vs-all (queries == candidates, no top-k).  Every rank holds the whole corpus and calls
 * wealy_eval_sweep_shard with its (shard_rank, shard_world): the symmetric sweep is restricted to the row blocks
 * rb = shard_rank (mod shard_world) and leaves this rank's share of the rank counts in the plan.  The caller
 * then sums the `count` uint32 values at `counts` over the ranks (one NCCL all-reduce) and calls
 * wealy_eval_finish, which yields the complete per-query AP / R1 / sums on every rank.                */
int wealy_eval_sweep_shard(wealy_eval_plan* plan, const void* z, int64_t ld, int64_t d, int dtype, float eps,
                           int passes, int shard_rank, int shard_world, void* stream);
int wealy_eval_plan_counts(const wealy_eval_plan* plan, void** counts, int64_t* count);
/* The sharded sweep in two stages: the relevant similarities (the thresholds the ranks are counted against) are computed
 * once ACROSS the ranks instead of once per rank.  _prepare: normalise + split the whole corpus, thresholds of this
 * rank's share of the queries (zeros elsewhere); the caller sums the `count` floats at `values`
 * (wealy_eval_plan_thresholds) over the ranks -- every element has exactly one non-zero contribution, so the sum is
 * exact --; _sweep: the rank's row blocks, as wealy_eval_sweep_shard; then counts / finish as above.            */
int wealy_eval_shard_prepare(wealy_eval_plan* plan, const void* z, int64_t ld, int64_t d, int dtype, float eps, int passes,
                             int shard_rank, int shard_world, void* stream);
int wealy_eval_plan_thresholds(const wealy_eval_plan* plan, void** values, int64_t* count);
int wealy_eval_shard_sweep(wealy_eval_plan* plan, int64_t d, int passes, int shard_rank, int shard_world, void* stream);
/* Multi-GPU all-vs-all of CHUNKED tracks (z [n * chunks, d], chunks in {2, 4, 8, 16}, redux WEALY_REDUX_*; lens NULL for
 * full tracks, else the device int32 [n] ragged chunk counts, used for both sides as in wealy_eval_run_ragged).  The
 * same protocol as above: every rank sweeps the row blocks rb = shard_rank (mod shard_world) of the chunked sweep --
 * the half sweep for min / max / mean, the rectangle for meanmin / minmean (or WEALY_SYM_TRACKS=0) -- then the counts
 * are summed over the ranks and wealy_eval_finish yields the per-track AP / R1.  No top-k; queries must be the
 * candidates (WEALY_ERR_BAD_ARG otherwise), other chunk counts WEALY_ERR_UNSUPPORTED.
 * Staged form: _prepare_tracks computes the relevant track similarities of this rank's contiguous share of the query
 * tracks, [n r / w, n (r + 1) / w), into a zeroed buffer; after _prepare_tracks, wealy_eval_plan_thresholds returns that
 * buffer alone: `count` = total_pairs floats, query q's sorted thresholds at [offsets[q], offsets[q + 1]) of
 * wealy_eval_plan_ranks' CSR offsets (after the vector _prepare it returns {lowest thresholds, all thresholds}).  The
 * caller sums it over the ranks; _sweep_tracks rebuilds the per-query counts and limits from it on every rank, then
 * sweeps the rank's row blocks.  d / passes / chunks / redux / lens of the two stages must agree. */
int wealy_eval_sweep_shard_tracks(wealy_eval_plan* plan, const void* z, int64_t ld, int64_t d, int dtype, float eps,
                                  int passes, int chunks, int redux, const int32_t* lens, int shard_rank, int shard_world,
                                  void* stream);
int wealy_eval_shard_prepare_tracks(wealy_eval_plan* plan, const void* z, int64_t ld, int64_t d, int dtype, float eps,
                                    int passes, int chunks, int redux, const int32_t* lens, int shard_rank, int shard_world,
                                    void* stream);
int wealy_eval_shard_sweep_tracks(wealy_eval_plan* plan, int64_t d, int passes, int chunks, int redux, const int32_t* lens,
                                  int shard_rank, int shard_world, void* stream);
/* Multi-GPU all-vs-all WITH top-k lists (plain [n, d] embeddings, queries == candidates).  Every rank calls
 * wealy_eval_sweep_shard_topk: the normalisation, the relevant similarities and the sampled per-query bounds of the
 * single-GPU symmetric top-k sweep run on every rank (identical on all of them), then the symmetric top-k sweep over the
 * row blocks rb = shard_rank (mod shard_world).  The rank counts stay in the plan (sum them over the ranks, then
 * wealy_eval_finish, as above); the rank's candidate lists are finalized locally: val / idx [n][k] (device float32 /
 * int32, the caller's row q, caller indices) hold the min(k, m) best of query q's m local candidates, by descending
 * similarity, ties to the lower index, padded with (-inf, -1); cnt [n] = m, or -1 where the list overflowed.  A list
 * shorter than k is no failure: the other ranks hold the rest.  WEALY_ERR_UNSUPPORTED, before any work, unless the
 * single-GPU call would take the symmetric top-k sweep (same ids, k <= 128, n >= max(WEALY_SYM_TOPK_MIN_ROWS, 192 k),
 * WEALY_SYM_TOPK != 0) and shard_world * k <= 1024; the decision reads only the arguments and the plan's ids, so every
 * rank reaches the same one.  wealy_eval_plan_last_topk_path reports 1, stage_ms' top-k finalize the local finalize.
 * wealy_eval_topk_merge then merges, per query, the lists of all ranks -- val / idx [world][n][k], cnt [world][n], as
 * sweep_shard_topk wrote them, each restricted to the same n queries (rank r typically receives every rank's rows of
 * its own query slice) -- into out_idx (int64) / out_sim [n][k]: the k best of the world * k entries, by descending
 * similarity, ties to the lower index, whatever the order of the world lists.  It ADDS to the device int32 *fail the
 * number of queries with a count of -1 or counts summing to less than k; for those the lists do not hold the k best,
 * and the caller recomputes them (e.g. with queries partitioned over the ranks).  k <= 128, world * k <= 1024. */
int wealy_eval_sweep_shard_topk(wealy_eval_plan* plan, const void* z, int64_t ld, int64_t d, int dtype, float eps,
                                int passes, int k, int shard_rank, int shard_world, float* val, int32_t* idx, int32_t* cnt,
                                void* stream);
int wealy_eval_topk_merge(const float* val, const int32_t* idx, const int32_t* cnt, int world, int64_t n, int k,
                          int64_t* out_idx, float* out_sim, int32_t* fail, void* stream);
int wealy_eval_finish(wealy_eval_plan* plan, float* aps, float* r1s, double* sums, void* stream);
/* Per-item ranks of the last run -- the quantities AP and R1 are made of.  offsets [nq + 1] int64 (CSR over the
 * caller's queries; offsets[nq] = total_pairs of wealy_eval_plan_info), ranks / sims [total_pairs]: for every query its
 * relevant candidates best first, rank = 1 + #{non-self candidates with a larger similarity}, sim = cosine similarity.
 * After a sharded sweep call it once the counters have been summed over the ranks.                             */
int wealy_eval_plan_ranks(const wealy_eval_plan* plan, int64_t* offsets, int32_t* ranks, float* sims, void* stream);
/* device time (CUDA events on the run's stream) of the fused similarity+ranking sweep of the last
 * wealy_eval_run on this plan; blocks until that sweep has finished.                           */
int wealy_eval_plan_last_sweep_ms(const wealy_eval_plan* plan, float* ms);
/* which kernel produced the top-k lists of the last run: 0 none, 1 the symmetric sweep (all-vs-all, N >= max(16384, 192 k),
 * k <= 128: sampled per-query bounds, candidates collected in both directions; synchronises the stream once to read a
 * 4-byte overflow flag), 2 the rectangle sweep with its streaming top-k, 3 = 1 failed its check and 2 recomputed.  */
int wealy_eval_plan_last_topk_path(const wealy_eval_plan* plan, int* path);
/* the same for the stages of the last run: ms[5] = {prep (normalise + fp16 split), K_pos (relevant similarities +
 * counter reset), fused sweep, ap_reduce, top-k finalize}; the last two are 0 after wealy_eval_sweep_shard, ap_reduce
 * is 0 after wealy_eval_sweep_shard_topk.  */
int wealy_eval_plan_stage_ms(const wealy_eval_plan* plan, float* ms);
void wealy_eval_plan_destroy(wealy_eval_plan* plan);

/* ---- a3: masked reductions ---------------------------------------------------------------
 * Replaces lib/tensor_ops.py:182-258 (msum / mmean / mmin / mmax): x [rows, cols] contiguous, reduced
 * over cols; mask [rows, cols] bytes, non-zero = EXCLUDED (may be NULL); out [rows] in x's dtype.
 * fill: value substituted for excluded entries in min / max (the reference's `ctt`); eps: the clamp
 * of the mean's denominator.  One HBM pass.                                                     */
#define WEALY_MASKED_SUM 0
#define WEALY_MASKED_MEAN 1
#define WEALY_MASKED_MIN 2
#define WEALY_MASKED_MAX 3
int wealy_masked_reduce(const void* x, const uint8_t* mask, int64_t rows, int64_t cols, int dtype, int op, float fill,
                        float eps, void* out, void* stream);
/* Gradient of wealy_masked_reduce: dx [rows, cols] (x's dtype) = g[row] * w, g [rows] in x's dtype, the same x / mask /
 * op / fill / eps as the forward.  w: sum 1, mean 1 / max(count, eps) on included entries (0 on excluded ones); min / max
 * with full == 0: 1 on the FIRST extreme of the filled row (a NaN is the extreme; 0 if that entry is excluded) -- order
 * the columns so that the reference's tie (the last dim it reduces is the most significant) is the first; full != 0
 * (dim=None, torch.min() of the whole tensor): 1 / t on every included entry equal to the extreme, t = the number of
 * positions equal to it, excluded ones counted.                                                                    */
int wealy_masked_reduce_backward(const void* x, const uint8_t* mask, int64_t rows, int64_t cols, int dtype, int op,
                                 float fill, float eps, int full, const void* g, void* dx, void* stream);

/* ---- a4: multi-chunk distance reduction -----------------------------------------------------
 * Replaces lib/tensor_ops.py:288-373 `distance_tensor_redux(dist, redux, mask, ...)`: dist [pairs, s1, s2] contiguous
 * (the (b1, b2) leading dimensions flattened), mask [pairs, s1, s2] bytes (non-zero = EXCLUDED; may be NULL), out [pairs]
 * in dist's dtype; s1, s2 <= 32.  op / karg: the strategy ("best-k" / "worst-k": k; "bpwr-n": n, 0 = all rounds;
 * for WEALY_RDX_BPWR the caller adds the reference's eps * rand tie-jitter to dist beforehand); symmetric != 0: the
 * "s" prefix (mean of the strategy on the block and on its transpose); eps: clamp of the means' denominators;
 * inf: the reference's `inf` stand-in (1e12).  "randmin" needs a random stream and stays a composition on the caller's side. */
#define WEALY_RDX_MIN 0
#define WEALY_RDX_MAX 1
#define WEALY_RDX_MEAN 2
#define WEALY_RDX_MINMEAN 3
#define WEALY_RDX_MEANMIN 4
#define WEALY_RDX_BEST 5
#define WEALY_RDX_WORST 6
#define WEALY_RDX_BPWR 7
int wealy_distance_redux(const void* dist, const uint8_t* mask, int64_t pairs, int s1, int s2, int dtype, int op, int karg,
                         int symmetric, float eps, float inf, void* out, void* stream);
/* Gradient of wealy_distance_redux: ddist [pairs, s1, s2] (dist's dtype) = g[pair] * w, g [pairs] in dist's dtype, the
 * same dist (for WEALY_RDX_BPWR the jittered one the forward saw) / mask / op / karg / symmetric / eps / inf.  The
 * strategy's selection is rerun; w is what the reference's autograd gives (DESIGN.md section 1, row a4): min / max
 * one-hot on the first extreme in row-major order, mean 1 / max(count, eps), minmean 1 / max(cnt_i, eps) on the first
 * minimal row, meanmin cnt_i / max(C, eps) on every row's first argmin, best-k / bpwr 1 / max(c, eps) on the selected
 * entries, worst-k 0; excluded entries 0; symmetric: the mean of the weights of the block and of its transpose.     */
int wealy_distance_redux_backward(const void* dist, const uint8_t* mask, int64_t pairs, int s1, int s2, int dtype, int op,
                                  int karg, int symmetric, float eps, float inf, const void* g, void* ddist, void* stream);

/* ---- f3 / f4: the steps either side of the path (SURVEY.md section 8(f)) --------------------------
 * wealy_mean_pool: lib/layers.py:6-30 MeanPool.  x [b, c, t] contiguous, mask [b, t] bytes (non-zero = VALID) or
 *   NULL; backward == 0: out [b, c] = masked temporal mean; backward != 0: x is the upstream gradient [b, c] and
 *   out [b, c, t] receives d/dx.
 * wealy_segment_mean: the avg-pool collate (lib/embedding_dataset/collate_functions.py:131-172, emb.mean(dim=0)):
 *   x [sum_T, dim] = the tracks' frames concatenated, offsets [tracks + 1] int64 -> out [tracks, dim] fp32.
 * wealy_triplet_mine: lib/losses.py:140-171 `_create_triplets`: positives[i] / negatives[i] = first index with
 *   the same label and a different idx / a different label, -1 if none.                                 */
int wealy_mean_pool(const void* x, const uint8_t* mask, int64_t b, int64_t c, int64_t t, int dtype, void* out,
                    int backward, void* stream);
int wealy_segment_mean(const void* x, const int64_t* offsets, int64_t tracks, int64_t dim, int dtype, float* out,
                       void* stream);
int wealy_triplet_mine(const int64_t* z_label, const int64_t* z_idx, int64_t b, int64_t* positives,
                       int64_t* negatives, void* stream);
/* wealy_triplet_forward / _backward: lib/losses.py:76-137 (torch.nn.TripletMarginLoss on the mined triplets).
 *   d(x, y) = ||x - y + eps||_p;  l_i = max(margin + d(a,p) - d_neg, 0), d_neg = d(a,n) or min(d(a,n), d(p,n)) (swap).
 *   forward: rows [b][4] f32 = (d_ap, d_an, d_pn, l_i; l_i = -1 for anchors without a triplet), acc[2] doubles =
 *   (sum of l_i, number of triplets).  backward: dz [b][d] fp32 (zeroed by the call) = sum_i g_i dl_i/dz with
 *   g_i = upstream[0] (/ number of triplets if `mean`) or upstream[i] if `per_anchor`.                      */
int wealy_triplet_forward(const void* z, int64_t ldz, int64_t b, int64_t d, int dtype, const int64_t* positives,
                          const int64_t* negatives, float margin, float p, float eps, int swap, float* rows,
                          double* acc, void* stream);
int wealy_triplet_backward(const void* z, int64_t ldz, int64_t b, int64_t d, int dtype, const int64_t* positives,
                           const int64_t* negatives, float p, float eps, int swap, const float* rows,
                           const float* upstream, int per_anchor, int mean, const double* acc, float* dz, void* stream);

/* ---- a5/a6: batch similarity-matrix contrastive losses -------------------------------------
 * NT-Xent: lib/losses.py:19-73.  CLEWS: lib/losses.py:210-285.  Forward writes the loss terms
 * and logdict statistics into `out` (doubles, device) and keeps the per-row statistics the
 * backward needs inside `workspace`; backward writes d loss / d z (dtype of z) scaled by
 * *grad_out (a device float, the upstream gradient of the scalar loss).
 *   z [b, d] (row stride ldz), z_label / z_idx [b] int64 (already label-noised by the caller,
 *   lib/losses.py:34-35).                                                                      */
#define WEALY_LOSS_NTXENT 0
#define WEALY_LOSS_CLEWS 1

/* indices into `out` */
#define WEALY_OUT_LOSS 0
#define WEALY_OUT_ZMAX 1
#define WEALY_OUT_ZMEAN 2
#define WEALY_OUT_ZSTD 3
#define WEALY_OUT_ALIGN 4     /* CLEWS l_cent */
#define WEALY_OUT_UNIFORM 5   /* CLEWS l_cont */
#define WEALY_OUT_NPOS 6      /* cnt_pos_pairs */
#define WEALY_OUT_NNEG 7      /* cnt_neg_pairs */
#define WEALY_OUT_ANCHORS 8   /* anchors_with_pos */
#define WEALY_OUT_DPOS 9      /* v_dpos */
#define WEALY_OUT_DNEG 10     /* v_dneg */
#define WEALY_OUT_BAD_IDS 11  /* number of z_label / z_idx values that do not fit in 32 bits; non-zero => loss is NaN */
#define WEALY_OUT_COUNT 16

typedef struct wealy_loss_cfg {
  int kind;          /* WEALY_LOSS_* */
  int passes;        /* WEALY_PASSES_* */
  float temperature; /* NT-Xent tau */
  float gamma, b;    /* CLEWS */
  float eps, epsilon;
  float uw;          /* CLEWS resolved uniformity weight */
  int numerically_friendly;
  int label_noise;   /* forward: apply lib/losses.py:34-35 inside the call -- a batch with a single label gets its first
                        max(2, b / 100) labels overwritten with -1 IN PLACE (single-GPU entry point, b <= 65536) */
  int grad_dtype;    /* backward: element type of *grad_out (WEALY_F32 / F16 / BF16) */
} wealy_loss_cfg;

size_t wealy_loss_workspace_bytes(int64_t b, int64_t d, int passes);
/* out: WEALY_OUT_COUNT doubles (all written); out_cast (nullable): the same numbers in z's element type -- what the
 * reference's modules hand back (loss and logdict carry z's dtype, lib/losses.py:65-72).  z_label is written only
 * when cfg->label_noise is set.  grad_out: one element of type cfg->grad_dtype.                                  */
int wealy_loss_forward(const wealy_loss_cfg* cfg, const void* z, int64_t b, int64_t ldz, int64_t d, int dtype,
                       int64_t* z_label, const int64_t* z_idx, double* out, void* out_cast, void* workspace,
                       size_t workspace_bytes, void* stream);
int wealy_loss_backward(const wealy_loss_cfg* cfg, const void* z, int64_t b, int64_t ldz, int64_t d, int dtype,
                        const void* grad_out, void* dz, int64_t ld_dz, void* workspace, size_t workspace_bytes,
                        void* stream);

/* ---- f2: data-parallel losses (global-batch NT-Xent / CLEWS over the GPUs of one box; not in the reference, which is
 * single-process -- SURVEY.md section 8(f)).  z / z_label / z_idx are the GLOBAL batch [b_global] (all-gathered by the
 * caller over NCCL), this rank owns the anchors [row0, row0 + nb).
 *   1. wealy_loss_dp_forward_local : prep of all rows, statistics sweep of this rank's anchors against all columns
 *   2. caller: all-reduce `acc` (count_acc doubles, SUM) and `acc_max` (2 x uint32, MAX), all-gather `rowstat`
 *      (4 floats per anchor; this rank wrote rows [row0, row0 + nb)) -- pointers from wealy_loss_dp_buffers
 *   3. wealy_loss_dp_forward_finish: loss terms + logdict statistics of the GLOBAL batch into `out` (same on all ranks)
 *   4. wealy_loss_dp_backward      : dz_rows [nb][d] = d(global loss)/dz of this rank's rows -- complete (the
 *      symmetrised dL/dS carries the terms in which these rows are columns of other ranks' anchors): no reduce-scatter. */
size_t wealy_loss_dp_workspace_bytes(int64_t b_global, int64_t d, int passes, int64_t nb);
int wealy_loss_dp_forward_local(const wealy_loss_cfg* cfg, const void* z, int64_t b_global, int64_t ldz, int64_t d,
                                int dtype, const int64_t* z_label, const int64_t* z_idx, int64_t row0, int64_t nb,
                                void* workspace, size_t workspace_bytes, void* stream);
/* wealy_loss_dp_forward_local split in two, so that the exchange of z overlaps the first part of the sweep: phase 1 reads
 * only this rank's own rows [row0, row0 + nb) of z (ids of the whole batch must be there) and sweeps its anchors against
 * its own column block; phase 2 -- once the all-gather has delivered the other rows -- preps them and sweeps the rest. */
int wealy_loss_dp_forward_phase(const wealy_loss_cfg* cfg, const void* z, int64_t b_global, int64_t ldz, int64_t d, int dtype,
                                const int64_t* z_label, const int64_t* z_idx, int64_t row0, int64_t nb, int phase,
                                void* workspace, size_t workspace_bytes, void* stream);
int wealy_loss_dp_buffers(const wealy_loss_cfg* cfg, void* workspace, size_t workspace_bytes, int64_t b_global, int64_t d,
                          int64_t nb, double** acc, int64_t* count_acc, uint32_t** acc_max, float** rowstat);
/* Step 2 as ONE collective for equal shards (rank r owns anchors [r nb, (r + 1) nb)): wealy_loss_dp_pack writes this
 * rank's {acc, acc_max, rowstat rows} into `record` (wealy_loss_dp_record_bytes(nb) bytes), the caller all-gathers the
 * records in rank order, wealy_loss_dp_unpack folds `world` of them back into the workspace (sums, maxima, all rows). */
size_t wealy_loss_dp_record_bytes(int64_t nb);
int wealy_loss_dp_pack(const wealy_loss_cfg* cfg, void* workspace, size_t workspace_bytes, int64_t b_global, int64_t d,
                       int64_t row0, int64_t nb, void* record, void* stream);
int wealy_loss_dp_unpack(const wealy_loss_cfg* cfg, void* workspace, size_t workspace_bytes, int64_t b_global, int64_t d,
                         int64_t nb, const void* records, int world, void* stream);
int wealy_loss_dp_forward_finish(const wealy_loss_cfg* cfg, int64_t b_global, int64_t d, int64_t nb, double* out,
                                 void* out_cast, int cast_dtype, void* workspace, size_t workspace_bytes, void* stream);
int wealy_loss_dp_backward(const wealy_loss_cfg* cfg, const void* z, int64_t b_global, int64_t ldz, int64_t d, int dtype,
                           int64_t row0, int64_t nb, const void* grad_out, void* dz_rows, int64_t ld_dz, void* workspace,
                           size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* WEALY_B200_H_ */
