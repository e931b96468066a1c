// Epilogue policies plugged into gemm_core.cuh.  Each thread owns ONE accumulator row (one query)
// and receives its similarities 32 consecutive candidates at a time, straight from TMEM.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "gemm_core.cuh"

namespace wealy {

// ---------------------------------------------------------------------------------------------
// StoreEpi: materialise the (n, m) matrix -- pairwise_distance_matrix (lib/tensor_ops.py:152-176)
// and pairwise_euclidean_distance_matrix (:131-149).  HBM-write bound; used for the drop-in
// `pairwise_distance_matrix` call and as the debug view of the fused kernels.
// ---------------------------------------------------------------------------------------------
enum SimMode : int {
  kSimCossim = 0,  // s                      (inputs pre-normalised by prep)
  kSimCos = 1,     // 1 - s
  kSimDotsim = 2,  // s * rs * cs            (power-of-two row scales folded back)
  kSimDot = 3,     // 1 - s * rs * cs
  kSimSqeuc = 4,   // max(|x|^2 - 2 x.y + |y|^2, 0) * post
  kSimEuc = 5,     // sqrt(max(..., 0)) * post
};

enum OutDtype : int { kOutF32 = 0, kOutF16 = 1, kOutBF16 = 2 };

struct StoreParams {
  void* out;
  long long ld;       // elements between consecutive output rows
  int mode;
  int out_dtype;
  float post;         // post scale (1/D for nsqeuc, D^-1/2 for neuc/nfro)
  const float* rscale;  // [n] row factors (RAW modes) or nullptr
  const float* cscale;  // [m]
  const float* rsq;     // [n] squared norms (euclidean modes)
  const float* csq;     // [m]
};

struct StoreEpi {
  using Params = StoreParams;
  static constexpr int kWarpScratchBytes = 0;
  static constexpr int kCtaScratchBytes = 0;
  struct RowState {
    float rs, rq;
    bool valid;
  };

  __device__ static __forceinline__ void row_begin(const Params& p, RowState& st, int row, int, const GemmShape& sh, const EpiCtx&) {
    st.valid = row < sh.m_rows;
    st.rs = (st.valid && p.rscale) ? p.rscale[row] : 1.f;
    st.rq = (st.valid && p.rsq) ? p.rsq[row] : 0.f;
  }

  __device__ static __forceinline__ float transform(const Params& p, const RowState& st, float s, int col) {
    switch (p.mode) {
      case kSimCossim: return s;
      case kSimCos: return 1.f - s;
      case kSimDotsim: return s * st.rs * (p.cscale ? __ldg(p.cscale + col) : 1.f);
      case kSimDot: return 1.f - s * st.rs * __ldg(p.cscale + col);
      default: {
        const float dot = s * st.rs * __ldg(p.cscale + col);
        float d2 = st.rq - 2.f * dot + __ldg(p.csq + col);
        d2 = d2 <= 0.f ? 0.f : d2;
        return (p.mode == kSimSqeuc ? d2 : sqrtf(d2)) * p.post;
      }
    }
  }

  __device__ static __forceinline__ void chunk32(const Params& p, RowState& st, int row, int col0,
                                                 const uint32_t (&acc)[32], const GemmShape& sh, const EpiCtx&) {
    if (!st.valid || col0 >= sh.n_cols) return;
    const int ncol = min(32, sh.n_cols - col0);
    float o[32];
#pragma unroll
    for (int e = 0; e < 32; ++e) o[e] = e < ncol ? transform(p, st, __uint_as_float(acc[e]), col0 + e) : 0.f;
    const long long base = (long long)row * p.ld + col0;
    if (p.out_dtype == kOutF32) {
      float* dst = reinterpret_cast<float*>(p.out) + base;
      if (ncol == 32 && ((reinterpret_cast<uintptr_t>(dst) & 15) == 0)) {
#pragma unroll
        for (int e = 0; e < 32; e += 4) *reinterpret_cast<float4*>(dst + e) = make_float4(o[e], o[e + 1], o[e + 2], o[e + 3]);
      } else {
#pragma unroll
        for (int e = 0; e < 32; ++e)
          if (e < ncol) dst[e] = o[e];
      }
    } else if (p.out_dtype == kOutF16) {
      __half* dst = reinterpret_cast<__half*>(p.out) + base;
#pragma unroll
      for (int e = 0; e < 32; ++e)
        if (e < ncol) dst[e] = __float2half_rn(o[e]);
    } else {
      __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(p.out) + base;
#pragma unroll
      for (int e = 0; e < 32; ++e)
        if (e < ncol) dst[e] = __float2bfloat16_rn(o[e]);
    }
  }

  __device__ static __forceinline__ void tile_begin(const Params&, RowState&, const GemmShape&, const EpiCtx&, int) {}
  __device__ static __forceinline__ void tile_end(const Params&, RowState&, const GemmShape&, const EpiCtx&) {}
  __device__ static __forceinline__ void row_end(const Params&, RowState&, int, int, const GemmShape&, const EpiCtx&) {}
};

// ---------------------------------------------------------------------------------------------
// EvalEpi: fused self / same-clique masking + rank counting (+ streaming top-k candidates).
// The evaluator is absent from the reference (SURVEY.md 8(a7)); semantics follow
// lib/losses.py:40-42 (ids, not positions) and lib/audio_dataset/dataset.py:82-86.
//
// Per query q the plan provides its P_q relevant similarities sorted ascending (thr) and
// lim_q = thr[0].  A candidate j that is neither self (i_j == i_q) nor relevant (c_j == c_q)
// and has s_qj > lim_q is binned by the number of thresholds below it:
//     hist[q][k-1] += 1,   k = #{p : thr_p < s_qj}  (k >= 1)
// so that  #{negatives above thr_r} = sum_{k > r} hist[q][k-1]  -- ranks without any sort and
// without the N x N matrix ever leaving the SM.  The overwhelmingly common case (s <= lim_q)
// costs one max-reduction over the 32-column chunk and one compare.
// ---------------------------------------------------------------------------------------------
// ---------------------------------------------------------------------------------------------
// warp_select_topk: in-place selection of the k largest of n (value, index) entries by one warp,
// O(n) work: the entries live in registers (kPerLane per lane), the k-th largest key is found by
// a 32-step bisection on the order-preserving integer image of the floats (one __reduce_add_sync
// per step), survivors are scattered to [0, k) (unsorted).  Requires k <= n <= 32 * kPerLane.
// Returns the k-th largest value.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned float_order_key(float f) {
  const unsigned b = __float_as_uint(f);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float float_from_order_key(unsigned k) {
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

template <int kPerLane>
__device__ __forceinline__ float warp_select_topk(float* val, int* idx, int n, int k, int lane) {
  constexpr unsigned kFull = 0xffffffffu;
  __syncwarp();  // entries appended by other lanes must be visible
  unsigned key[kPerLane];
  int id[kPerLane];
#pragma unroll
  for (int j = 0; j < kPerLane; ++j) {
    const int e = j * 32 + lane;
    const bool ok = e < n;
    key[j] = ok ? float_order_key(val[e]) : 0u;  // 0 is below the key of every float
    id[j] = ok ? idx[e] : -1;
  }
  unsigned T = 0;
  for (int b = 31; b >= 0; --b) {
    const unsigned cand = T | (1u << b);
    int c = 0;
#pragma unroll
    for (int j = 0; j < kPerLane; ++j) c += key[j] >= cand;
    c = __reduce_add_sync(kFull, c);
    if (c >= k) T = cand;  // warp-uniform
  }
  int g = 0, q = 0;
#pragma unroll
  for (int j = 0; j < kPerLane; ++j) {
    g += key[j] > T;
    q += key[j] == T;
  }
  int gi = g, qi = q;  // inclusive scans over lanes
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int tg = __shfl_up_sync(kFull, gi, o);
    const int tq = __shfl_up_sync(kFull, qi, o);
    if (lane >= o) { gi += tg; qi += tq; }
  }
  const int G = __shfl_sync(kFull, gi, 31);
  int pg = gi - g;          // first slot of this lane's "greater" entries
  int pq = G + (qi - q);    // first slot of this lane's "equal" entries (kept while < k)
  __syncwarp();             // every lane holds its entries in registers before anything is overwritten
#pragma unroll
  for (int j = 0; j < kPerLane; ++j) {
    if (key[j] > T) {
      val[pg] = float_from_order_key(key[j]);
      idx[pg] = id[j];
      ++pg;
    } else if (key[j] == T && key[j] != 0u) {
      if (pq < k) {
        val[pq] = float_from_order_key(key[j]);
        idx[pq] = id[j];
      }
      ++pq;
    }
  }
  __syncwarp();
  return float_from_order_key(T);
}

// out-of-line variants for the long candidate lists of large k (keeps the sweep kernel's hot path lean)
template <int kPerLane>
__device__ __noinline__ float warp_select_topk_big(float* val, int* idx, int n, int k, int lane) {
  return warp_select_topk<kPerLane>(val, idx, n, k, lane);
}

// Streaming variant used while a sweep is running: the list only has to shrink to ABOUT k entries and the filter only
// has to be a lower bound of the k-th best, so the bisection stops as soon as at most k + kSlackTopk entries lie at
// or above the prefix found so far (16-20 of the 32 steps on similarity data; exact ties fall through to all 32).
// Keeps every entry above the prefix (plus entries equal to it up to k); returns the filter, *kept = survivors.
constexpr int kSlackTopk = 24;
template <int kPerLane>
__device__ __forceinline__ float warp_compact_topk(float* val, int* idx, int n, int k, int lane, int* kept) {
  constexpr unsigned kFull = 0xffffffffu;
  __syncwarp();
  unsigned key[kPerLane];
  int id[kPerLane];
#pragma unroll
  for (int j = 0; j < kPerLane; ++j) {
    const int e = j * 32 + lane;
    const bool ok = e < n;
    key[j] = ok ? float_order_key(val[e]) : 0u;
    id[j] = ok ? idx[e] : -1;
  }
  unsigned T = 0;
  int at_or_above = n;  // entries with key >= T
  for (int b = 31; b >= 0; --b) {
    const unsigned cand = T | (1u << b);
    int c = 0;
#pragma unroll
    for (int j = 0; j < kPerLane; ++j) c += key[j] >= cand;
    c = __reduce_add_sync(kFull, c);
    if (c >= k) { T = cand; at_or_above = c; }  // warp-uniform
    if (at_or_above <= k + kSlackTopk) break;
  }
  int g = 0, q = 0;
#pragma unroll
  for (int j = 0; j < kPerLane; ++j) {
    g += key[j] > T;
    q += key[j] == T;
  }
  int gi = g, qi = q;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int tg = __shfl_up_sync(kFull, gi, o);
    const int tq = __shfl_up_sync(kFull, qi, o);
    if (lane >= o) { gi += tg; qi += tq; }
  }
  const int G = __shfl_sync(kFull, gi, 31), Q = __shfl_sync(kFull, qi, 31);
  const int limit = G > k ? G : k;  // entries equal to the prefix are kept while fewer than k survive
  int pg = gi - g;
  int pq = G + (qi - q);
  __syncwarp();
#pragma unroll
  for (int j = 0; j < kPerLane; ++j) {
    if (key[j] > T) {
      val[pg] = float_from_order_key(key[j]);
      idx[pg] = id[j];
      ++pg;
    } else if (key[j] == T && key[j] != 0u) {
      if (pq < limit) {
        val[pq] = float_from_order_key(key[j]);
        idx[pq] = id[j];
      }
      ++pq;
    }
  }
  __syncwarp();
  *kept = G + Q < limit ? G + Q : limit;
  return float_from_order_key(T);
}
template <int kPerLane>
__device__ __noinline__ float warp_compact_topk_big(float* val, int* idx, int n, int k, int lane, int* kept) {
  return warp_compact_topk<kPerLane>(val, idx, n, k, lane, kept);
}

struct EvalParams {
  const float* lim;        // [nq] lowest relevant similarity of the query (+inf if none)
  const int* q_c;          // [nq] clique ids
  const int* q_i;          // [nq] version ids
  const int* c_c;          // [nc]
  const int* c_i;          // [nc]
  const float* thr;        // CSR: sorted ascending relevant similarities
  const long long* off;    // [nq] CSR offsets
  const int* cnt;          // [nq] P_q
  unsigned int* hist;      // CSR, same indexing as thr
  // streaming top-k (k == 0 disables)
  int topk;
  int cap;                 // candidate-buffer capacity per (row, part)
  float* cand_val;         // [parts][nq][cap]
  int* cand_idx;
  int* cand_cnt;           // [parts][nq]
  int nq_total;
  // chunked tracks (SURVEY.md 8(f) row f1): kS consecutive rows / columns are the chunks of one track; a tile's
  // kS x kS blocks are reduced to one track-level similarity before ranking (distance_tensor_redux,
  // lib/tensor_ops.py:288-373, in similarity space: min distance = max similarity).  All arrays above are per TRACK.
  int red_inner, red_outer;  // kRedMax / kRedMin / kRedSum over the candidate's chunks, then over the query's
  float red_scale;           // 1, 1/kS or 1/kS^2 (means)
  // ragged tracks: valid chunks per query / candidate track (1 .. kS; chunks past the count are padding and are
  // excluded like distance_tensor_redux's mask, lib/tensor_ops.py:288; means divide by the valid counts); null = all kS
  const int* q_len;          // [nq]
  const int* c_len;          // [nc]
};

enum : int { kRedMax = 0, kRedMin = 1, kRedSum = 2 };

__device__ __forceinline__ float red_op(float a, float b, int op) {
  return op == kRedMax ? fmaxf(a, b) : (op == kRedMin ? fminf(a, b) : a + b);
}
__device__ __forceinline__ float red_neutral(int op) {
  return op == kRedMax ? __int_as_float(0xff800000) : (op == kRedMin ? __int_as_float(0x7f800000) : 0.f);
}

// kSym (chunked all-vs-all, queries == candidates, no top-k, a reduction that is the same in both directions): the
// sweep visits only the tiles that reach above the diagonal (GemmShape::sym on the CTA-pair core) and every track pair
// (q, c) with c > q is scored twice -- as candidate c of query q (the row direction: everything below, unchanged) and as
// candidate q of query c (the column direction: the lowest threshold of the chunk's 32 / kS column tracks is prefetched
// with their ids, the few elements that pass are queued with a direction bit and binned against the global CSR
// thresholds of their column query).
template <int kQueueCapT, int kCachePairsT, int kS = 1, bool kSym = false>
struct EvalEpiT {
  static_assert(kS == 1 || kS == 2 || kS == 4 || kS == 8 || kS == 16 || kS == 32, "chunks per track: a power of two <= 32");
  // tracks per 32-row / 32-column chunk.  kS = 32 (kGroups = 1): a warp's 32 rows are one query track and a chunk's 32
  // columns one candidate track -- the reduction over the candidate's chunks stays in the lane's 32 registers, the one
  // over the query's chunks takes the whole warp's shuffles, lane 0 carries the track's state, and every expression
  // below holds with a single group (64 chunks would put one track's rows in two epilogue warps)
  static constexpr int kGroups = 32 / kS;
  using Params = EvalParams;
  // Shared-memory scratch of the epilogue.
  //  * per warp, a work queue: the elements that pass the per-row limit are scattered unevenly over
  //    the 32 rows of a warp (a query with a poorly ranked relevant item passes almost everything,
  //    most queries pass nothing).  Handling them in place would serialise the warp on its hottest
  //    lane, so they are compacted into a queue and processed 32 at a time with every lane busy.
  //  * per CTA, a cache of the row block's thresholds: the CSR slice thr[off[row0] .. off[row0+128])
  //    is contiguous in global memory, so it is copied once per unit; each queued element is then
  //    binned by a binary search on shared memory (no dependent L2 round trips) and counted in a
  //    packed 16-bit shared-memory counter that is flushed to the global histogram at the end of
  //    the unit.  Rows whose thresholds do not fit (a row block concentrated in one giant clique)
  //    fall back to the global CSR arrays.
  static constexpr int kQueueCap = kQueueCapT;       // 256 with 8 epilogue warps, 128 with 16
  static constexpr int kBatchCols = kQueueCap / 32;  // columns per batch when a chunk overflows the queue
  static constexpr int kOffTag = kQueueCap * 4;
  static constexpr int kOffCand = kOffTag + kQueueCap * 2;
  static constexpr int kWarpScratchBytes = kOffCand + 32 * 4;
  static constexpr int kCachePairs = kCachePairsT;  // mean of a 128-row block is ~2100 on SHS100K-shaped data
  static constexpr int kCtaScratchBytes = kCachePairs * 6;
  static_assert(kCachePairs % 8 == 0, "cache regions stay 16-byte aligned");
  struct RowState {
    float lim;      // min(lowest threshold, top-k filter): the only compare on the fast path
    float tlim;     // lowest threshold
    float tau;      // top-k filter (k-th best so far, -inf until k candidates are buffered)
    int qc, qi, cnt;
    int so;         // offset of the row's thresholds inside the shared cache, -1 if not cached
    int n_cached;   // cached pairs of the unit (all threads hold the same value)
    int cc_next, ci_next, next_col;  // ids of this lane's column in the NEXT chunk (prefetched)
    float clim_next;                 // kSym: lowest threshold of that column's query
    float clim_q[4];                 // kSym: per queued chunk, like cc_q
    int own;                         // kSym: this lane carries a valid track
    long long off;
    long long base; // off[] of the unit's first row
    long long cbase;
    // deferred work: up to kSlots chunks are queued before the accumulator is released and drained after
    int qn, nslot;                       // queued elements / chunks (warp-uniform)
    int q_end[4], col0_q[4];             // per queued chunk: end of its queue range, first column (uniform)
    int cc_q[4], ci_q[4], ok_q[4];       // per queued chunk: ids / validity of this lane's column
  };
  static constexpr int kSlots = 4;

  __device__ static __forceinline__ float* q_val(const EpiCtx& c) { return reinterpret_cast<float*>(c.warp_scratch); }
  __device__ static __forceinline__ uint16_t* q_tag(const EpiCtx& c) {
    return reinterpret_cast<uint16_t*>(c.warp_scratch + kOffTag);
  }
  __device__ static __forceinline__ int* n_cand(const EpiCtx& c) { return reinterpret_cast<int*>(c.warp_scratch + kOffCand); }
  __device__ static __forceinline__ float* thr_s(const EpiCtx& c) { return reinterpret_cast<float*>(c.cta_scratch); }
  __device__ static __forceinline__ unsigned* cnt_s(const EpiCtx& c) {
    return reinterpret_cast<unsigned*>(c.cta_scratch + kCachePairs * 4);
  }
  __device__ static __forceinline__ void prefetch_ids(const Params& p, RowState& st, const GemmShape& sh, int lane) {
    const int col = st.next_col / kS + lane;  // candidate (track) this lane stands for in the next chunk
    const bool ok = lane < kGroups && col < sh.n_cols / kS;
    st.cc_next = ok ? __ldg(p.c_c + col) : 0;
    st.ci_next = ok ? __ldg(p.c_i + col) : 0;
    if constexpr (kSym) st.clim_next = ok ? __ldg(p.lim + col) : __int_as_float(0x7f800000);
  }

  __device__ static __forceinline__ void row_begin(const Params& p, RowState& st, int row, int part,
                                                   const GemmShape& sh, const EpiCtx& ctx) {
    const int lane = (int)ptx::lane_id();
    st.tlim = __int_as_float(0x7f800000);
    st.tau = __int_as_float(0x7f800000);
    st.qc = st.qi = st.cnt = 0;
    st.off = 0;
    const int q = row / kS;                                    // query (track) of this row
    const bool own = row < sh.m_rows && (lane % kS) == 0;      // one lane per track carries its state
    st.cbase = ((long long)part * p.nq_total + q) * p.cap;
    st.own = own;
    if (own) {
      st.tlim = p.lim[q];
      st.qc = p.q_c[q];
      st.qi = p.q_i[q];
      st.cnt = p.cnt[q];
      st.off = p.off[q];
      if (p.topk > 0) st.tau = __int_as_float(0xff800000);
    }
    st.lim = fminf(st.tlim, st.tau);
    st.next_col = ctx.first_col;
    st.qn = 0;
    st.nslot = 0;
    prefetch_ids(p, st, sh, lane);
    n_cand(ctx)[lane] = 0;
    // cooperative fill of the threshold cache (the previous unit's row_end left it flushed)
    // (the CTA-pair core may hand a CTA a row block that lies entirely past the last query)
    st.base = p.off[min(ctx.row_base, sh.m_rows) / kS];
    const long long total = p.off[min(ctx.row_base + kTileM, sh.m_rows) / kS] - st.base;
    st.n_cached = (int)(total < (long long)kCachePairs ? total : (long long)kCachePairs);
    float* ts = thr_s(ctx);
    unsigned* cs = cnt_s(ctx);
    for (int i = ctx.tid; i < st.n_cached; i += ctx.nthreads) ts[i] = __ldg(p.thr + st.base + i);
    for (int i = ctx.tid; i < (st.n_cached + 1) / 2; i += ctx.nthreads) cs[i] = 0u;
    const long long rel = st.off - st.base;
    st.so = (own && rel + st.cnt <= (long long)st.n_cached) ? (int)rel : -1;
    ptx::named_barrier_sync(1, ctx.nthreads);
  }

  // number of thresholds strictly below s (lower bound); thr[0 .. cnt) ascending
  __device__ static __forceinline__ int count_below(const float* __restrict__ thr, int cnt, float s) {
    int lo = 0, hi = cnt;
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (__ldg(thr + mid) < s) lo = mid + 1; else hi = mid;
    }
    return lo;
  }
  __device__ static __forceinline__ int count_below_smem(const float* thr, int cnt, float s) {
    // (a two-level pivot search with independent loads was measured 7 % slower than this plain
    // binary search: its extra address arithmetic and bank conflicts outweigh the shorter chain)
    int lo = 0, hi = cnt;
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (thr[mid] < s) lo = mid + 1; else hi = mid;
    }
    return lo;
  }

  __device__ static __forceinline__ int warp_incl_scan(int v, int lane) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, v, o);
      if (lane >= o) v += t;
    }
    return v;
  }

  // Process the queue range [begin, end): 32 elements per round, every lane busy.  cc / ci / colok are the
  // ids and validity of this lane's column in the chunk the range came from; col0 its first column.
  __device__ static __forceinline__ void process_range(const Params& p, RowState& st, const EpiCtx& ctx, int begin,
                                                       int end, int cc, int ci, int colok, int col0, int lane,
                                                       float clim = 0.f) {
    constexpr unsigned kFull = 0xffffffffu;
    const float* qv = q_val(ctx);
    const uint16_t* qt = q_tag(ctx);
    int* ncand = n_cand(ctx);
    const float* ts = thr_s(ctx);
    unsigned* cs = cnt_s(ctx);
    for (int r0 = begin; r0 < end; r0 += 32) {
      const int r = r0 + lane;
      const bool active = r < end;
      const float s = active ? qv[r] : 0.f;
      const int tag = active ? (int)qt[r] : 0;
      const int L = (tag >> 5) & 31, e = tag & 31;  // row lane and column of the element
      const bool coldir = kSym && (tag >> 10) != 0;  // the element scores its COLUMN's query (candidate: the row's track)
      const int rqc = __shfl_sync(kFull, st.qc, L);
      const int rqi = __shfl_sync(kFull, st.qi, L);
      const int rpc = __shfl_sync(kFull, st.cnt, L);
      const int rso = __shfl_sync(kFull, st.so, L);
      const float rtl = __shfl_sync(kFull, st.tlim, L);
      const float tau = __shfl_sync(kFull, st.tau, L);
      const int ccol = __shfl_sync(kFull, cc, e);
      const int cicol = __shfl_sync(kFull, ci, e);
      const int ok = __shfl_sync(kFull, colok, e);
      // i_j == i_q: self (or a version-id collision), never a candidate -- the test is symmetric
      const bool cand = active && ok && cicol != rqi;
      int pc = rpc, so = rso;
      float tl = rtl;
      if constexpr (kSym) {
        const float cl = __shfl_sync(kFull, clim, e);
        if (coldir) {
          tl = cl;
          so = -1;  // binned against the column query's thresholds in the global CSR
        }
      }
      if (cand && p.topk > 0 && s > tau) {
        const int slot = atomicAdd(&ncand[L], 1);
        const long long cb = st.cbase + (long long)(L / kS - lane / kS) * p.cap + slot;  // tracks of a warp are consecutive
        p.cand_val[cb] = s;
        p.cand_idx[cb] = col0 + e;
      }
      // rank counting: a negative above at least the lowest relevant item; k = #{thresholds < s} >= 1
      const bool neg = cand && s > tl && ccol != rqc;
      const bool cached = neg && so >= 0;
      int k = 0;
      if (cached) k = count_below_smem(ts + so, pc, s);
      // the elements of a round mostly come from one hot query and land in one bucket: the first
      // cached lane counts all lanes that share its (cache, bucket) key with a single shared-memory
      // atomic, the others add their own
      const int slot_idx = so + k - 1;
      const int key = cached ? slot_idx : -1;
      const unsigned cm = __ballot_sync(kFull, cached);
      if (cm != 0u) {
        const int lead = __ffs(cm) - 1;
        const int key_lead = __shfl_sync(kFull, key, lead);
        const unsigned same = __ballot_sync(kFull, cached && key == key_lead);
        if (cached && (lane == lead || key != key_lead)) {
          const unsigned add = lane == lead ? (unsigned)__popc(same) : 1u;
          const int shift = (slot_idx & 1) * 16;
          const unsigned old = (atomicAdd(cs + (slot_idx >> 1), add << shift) >> shift) & 0xffffu;
          // keep the 16-bit field far from overflow: the (single) adder that takes it across 0x8000
          // moves exactly 0x8000 counts to the global histogram
          if (old < 0x8000u && old + add >= 0x8000u) {
            atomicSub(cs + (slot_idx >> 1), 0x8000u << shift);
            atomicAdd(p.hist + st.base + slot_idx, 0x8000u);
          }
        }
      }
      const long long offL = __shfl_sync(kFull, st.off, L);
      if (neg && so < 0) {  // thresholds not cached (giant clique; column direction): global CSR arrays
        long long o = offL;
        if constexpr (kSym) {
          if (coldir) {
            o = __ldg(p.off + col0 + e);
            pc = __ldg(p.cnt + col0 + e);
          }
        }
        k = count_below(p.thr + o, pc, s);
        if (k > 0) atomicAdd(p.hist + o + (k - 1), 1u);
      }
    }
  }

  // top-k: a row gains at most 32 candidates per chunk; select its k best in place (warp-cooperatively,
  // one row at a time) as soon as fewer than kSlots * 32 free slots remain
  __device__ static __forceinline__ void compact_topk(const Params& p, RowState& st, const EpiCtx& ctx, int lane) {
    constexpr unsigned kFull = 0xffffffffu;
    int* ncand = n_cand(ctx);
    unsigned need = __ballot_sync(kFull, ncand[lane] > p.cap - kSlots * 32);
    while (need) {
      const int src = __ffs(need) - 1;
      need &= need - 1;
      const long long cb = st.cbase + (long long)(src / kS - lane / kS) * p.cap;
      const int n = ncand[src];
      int kept = p.topk;
      const float kth = p.cap <= 256   ? warp_compact_topk<8>(p.cand_val + cb, p.cand_idx + cb, n, p.topk, lane, &kept)
                        : p.cap <= 512 ? warp_compact_topk_big<16>(p.cand_val + cb, p.cand_idx + cb, n, p.topk, lane, &kept)
                                       : warp_compact_topk_big<32>(p.cand_val + cb, p.cand_idx + cb, n, p.topk, lane, &kept);
      if (lane == src) {
        ncand[lane] = kept;
        st.tau = kth;
        st.lim = fminf(st.tlim, st.tau);
      }
      __syncwarp();
    }
  }

  // Drain the deferred chunks (called after the accumulator has been handed back to the MMA warp).
  __device__ static __forceinline__ void drain(const Params& p, RowState& st, const EpiCtx& ctx) {
    if (st.nslot == 0) return;
    const int lane = (int)ptx::lane_id();
    __syncwarp();
    int begin = 0;
#pragma unroll
    for (int sl = 0; sl < kSlots; ++sl) {
      if (sl < st.nslot) {
        process_range(p, st, ctx, begin, st.q_end[sl], st.cc_q[sl], st.ci_q[sl], st.ok_q[sl], st.col0_q[sl], lane,
                      kSym ? st.clim_q[sl] : 0.f);
        begin = st.q_end[sl];
      }
    }
    __syncwarp();
    st.qn = 0;
    st.nslot = 0;
    if (p.topk > 0) compact_topk(p, st, ctx, lane);
  }

  // scatter the elements selected by `mb` into the queue starting at `base`; returns their number
  __device__ static __forceinline__ int push(const EpiCtx& ctx, const uint32_t (&acc)[32], unsigned mb, int base,
                                             int lane, int dir = 0) {
    float* qv = q_val(ctx);
    uint16_t* qt = q_tag(ctx);
    const int mine = __popc(mb);
    const int incl = warp_incl_scan(mine, lane);
    int pos = base + incl - mine;
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      // lukewarm chunks have a handful of passing elements: skip the 8-column groups nobody needs
      if (__any_sync(0xffffffffu, (mb & (0xffu << (8 * g))) != 0u)) {
#pragma unroll
        for (int e = 8 * g; e < 8 * g + 8; ++e) {
          if (mb & (1u << e)) {
            qv[pos] = __uint_as_float(acc[e]);
            qt[pos] = (uint16_t)((dir << 10) | (lane << 5) | e);
            ++pos;
          }
        }
      }
    }
    return __shfl_sync(0xffffffffu, incl, 31);
  }

  // kS x kS blocks of the chunk -> one similarity per (query track, candidate track): first over the candidate's
  // chunks (kS consecutive registers), then over the query's (kS adjacent lanes); entries >= kGroups are -inf
  __device__ static __forceinline__ void reduce_tracks(const Params& p, const uint32_t (&raw)[32], uint32_t (&out)[32],
                                                       int row, int col0, const GemmShape& sh) {
    if (p.c_len == nullptr) {
#pragma unroll
      for (int g = 0; g < kGroups; ++g) {
        float v = __uint_as_float(raw[g * kS]);
#pragma unroll
        for (int b = 1; b < kS; ++b) v = red_op(v, __uint_as_float(raw[g * kS + b]), p.red_inner);
        if (p.red_inner == kRedSum && p.red_outer != kRedSum) v *= p.red_scale;  // mean over the candidate's chunks first
#pragma unroll
        for (int o = 1; o < kS; o <<= 1) v = red_op(v, __shfl_xor_sync(0xffffffffu, v, o), p.red_outer);
        if (p.red_outer == kRedSum) v *= p.red_scale;
        out[g] = __float_as_uint(v);
      }
    } else {
      // ragged tracks: chunks past a track's count never enter a reduction (selects, so padding may hold anything)
      const int lane = (int)ptx::lane_id();
      const int tc = col0 / kS + lane;
      const int lq = row < sh.m_rows ? min(max(__ldg(p.q_len + row / kS), 1), kS) : kS;
      const int lc_mine = (lane < kGroups && tc < sh.n_cols / kS) ? min(max(__ldg(p.c_len + tc), 1), kS) : kS;
      const bool q_ok = (row & (kS - 1)) < lq;
      const float rq = 1.f / (float)lq, neutral = red_neutral(p.red_outer);
#pragma unroll
      for (int g = 0; g < kGroups; ++g) {
        const int lc = __shfl_sync(0xffffffffu, lc_mine, g);
        float v = __uint_as_float(raw[g * kS]);
#pragma unroll
        for (int b = 1; b < kS; ++b) v = b < lc ? red_op(v, __uint_as_float(raw[g * kS + b]), p.red_inner) : v;
        if (p.red_inner == kRedSum) v *= 1.f / (float)lc;
        v = q_ok ? v : neutral;
#pragma unroll
        for (int o = 1; o < kS; o <<= 1) v = red_op(v, __shfl_xor_sync(0xffffffffu, v, o), p.red_outer);
        if (p.red_outer == kRedSum) v *= rq;
        out[g] = __float_as_uint(v);
      }
    }
#pragma unroll
    for (int g = kGroups; g < 32; ++g) out[g] = 0xff800000u;
  }

  __device__ static __forceinline__ void chunk32(const Params& p, RowState& st, int row, int col0,
                                                 const uint32_t (&acc)[32], const GemmShape& sh, const EpiCtx& ctx) {
    if constexpr (kS > 1) {
      uint32_t red[32];
      reduce_tracks(p, acc, red, row, col0, sh);
      chunk32_tracks(p, st, row, col0 / kS, red, sh, ctx);
    } else {
      chunk32_tracks(p, st, row, col0, acc, sh, ctx);
    }
  }

  // col0: first candidate (track) of the chunk; acc[e] = similarity of this lane's query and candidate col0 + e
  __device__ static __forceinline__ void chunk32_tracks(const Params& p, RowState& st, int row, int col0,
                                                        const uint32_t (&acc)[32], const GemmShape& sh, const EpiCtx& ctx) {
    constexpr unsigned kFull = 0xffffffffu;
    const int lane = (int)ptx::lane_id();
    // ids of the 32 candidates of this chunk, one per lane, were prefetched during the previous
    // chunk; start the loads for the next one now so their L2 latency is off the critical path
    const int cc = st.cc_next, ci = st.ci_next;
    const float clim = kSym ? st.clim_next : 0.f;
    const int colok = lane < kGroups && (col0 + lane) < sh.n_cols / kS;
    st.next_col = col0 * kS + ctx.col_step;
    prefetch_ids(p, st, sh, lane);

    // ---- fast path: one compare per element, nothing else when no lane of the warp passes
    unsigned m = 0, mc = 0;
#pragma unroll
    for (int e = 0; e < 32; ++e) m |= (__uint_as_float(acc[e]) > st.lim) ? (1u << e) : 0u;
    if constexpr (kSym) {
      // column direction: the element against the lowest threshold of its column's query; a pair is scored (both
      // ways) where it is met above the diagonal, c > q
#pragma unroll
      for (int e = 0; e < kGroups; ++e) {
        const float cl = __shfl_sync(kFull, clim, e);
        mc |= (__uint_as_float(acc[e]) > cl) ? (1u << e) : 0u;
      }
      const int d = row / kS - col0;
      const unsigned above = d < 0 ? 0xffffffffu : (d >= 31 ? 0u : (0xffffffffu << (d + 1)));
      m &= above;
      mc = st.own ? (mc & above) : 0u;
    }
    if (!__any_sync(kFull, (m | mc) != 0)) return;

    // ---- collect: the passing elements go to the warp queue; they are binned in drain(), after the
    // accumulator has been released, so the MMA warp never waits for a slow chunk
    const int total = __reduce_add_sync(kFull, __popc(m) + __popc(mc));
    if (st.nslot == kSlots || st.qn + total > kQueueCap) drain(p, st, ctx);
    if (total <= kQueueCap) {
      const int n_row = push(ctx, acc, m, st.qn, lane);
      if constexpr (kSym) push(ctx, acc, mc, st.qn + n_row, lane, 1);
      st.qn += total;
      const int sl = st.nslot++;
#pragma unroll
      for (int k = 0; k < kSlots; ++k) {
        if (k == sl) {
          st.q_end[k] = st.qn;
          st.col0_q[k] = col0;
          st.cc_q[k] = cc;
          st.ci_q[k] = ci;
          st.ok_q[k] = colok;
          if constexpr (kSym) st.clim_q[k] = clim;
        }
      }
    } else {
      // a chunk denser than the whole queue: bin it now, kBatchCols columns at a time
      constexpr int kCols = kBatchCols;
#pragma unroll 1
      for (int dir = 0; dir < (kSym ? 2 : 1); ++dir) {
#pragma unroll 1
        for (int bi = 0; bi < 32 / kCols; ++bi) {
          const unsigned sel = ((1u << kCols) - 1u) << (kCols * bi);
          const int n = push(ctx, acc, (dir ? mc : m) & sel, 0, lane, dir);
          __syncwarp();
          process_range(p, st, ctx, 0, n, cc, ci, colok, col0, lane, clim);
          __syncwarp();
        }
      }
      if (p.topk > 0) compact_topk(p, st, ctx, lane);
    }
    (void)row;
  }

  __device__ static __forceinline__ void tile_begin(const Params&, RowState&, const GemmShape&, const EpiCtx&, int) {}

  __device__ static __forceinline__ void tile_end(const Params& p, RowState& st, const GemmShape&, const EpiCtx& ctx) {
    drain(p, st, ctx);
  }

  __device__ static __forceinline__ void row_end(const Params& p, RowState& st, int row, int part,
                                                 const GemmShape& sh, const EpiCtx& ctx) {
    const int lane = (int)ptx::lane_id();
    if (p.topk > 0 && row < sh.m_rows && (lane % kS) == 0) p.cand_cnt[(long long)part * p.nq_total + row / kS] = n_cand(ctx)[lane];
    ptx::named_barrier_sync(1, ctx.nthreads);  // every warp has finished counting into the cache
    const unsigned* cs = cnt_s(ctx);
    for (int i = ctx.tid; i < st.n_cached; i += ctx.nthreads) {
      const unsigned v = (cs[i >> 1] >> ((i & 1) * 16)) & 0xffffu;
      if (v != 0u) atomicAdd(p.hist + st.base + i, v);
    }
    ptx::named_barrier_sync(1, ctx.nthreads);  // flushed before the next unit refills the cache
  }
};

using EvalEpi = EvalEpiT<256, 3456>;           // 8 epilogue warps
template <int kS>
using EvalTracksEpi = EvalEpiT<256, 3456, kS>;  // kS chunk embeddings per track, reduced in the epilogue
template <int kS>
using EvalTracksSymEpi = EvalEpiT<256, 3456, kS, true>;  // ... chunked all-vs-all: tiles above the diagonal, both directions

}  // namespace wealy
