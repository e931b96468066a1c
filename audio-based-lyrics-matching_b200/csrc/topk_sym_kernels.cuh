// Top-k inside the SYMMETRIC all-vs-all sweep (a7 with top-k output, e.g. BASELINE configs[4]: 50k x 2048, top-100).
//
// The rectangle sweep keeps a streaming top-k per (row, part) with a filter that tightens as the row's sweep
// advances; that needs every query to see ALL its candidates in its own row, i.e. the full N x N contraction.  The
// symmetric sweep contracts only the tiles above the diagonal and scores every element for its row query AND its
// column query, so a query's candidates arrive from many CTAs in no particular order.  What makes top-k possible
// there is a STATIC per-query lower bound beta_q of the k-th best similarity, known before the sweep starts:
//
//   1. sample:   S candidates, evenly spaced in clique-sorted order (S ~ N / 16, at least 4096);
//   2. pre-pass: every query against the sample in one fp16 pass (the bound does not have to be exact) with an epilogue
//                that keeps the maximum of every 32-column group; beta_q = the (r + 1)-th largest group maximum, a lower
//                bound of the sample's (r + 1)-th best, r = max(24, 3 k S / N): about 3 k candidates of the whole
//                corpus lie above it (relative spread of that count: 1 / sqrt(r));
//   3. sweep:    EvalSymEpi<..., kTopk = true> appends every element above beta_row / beta_col to the row's / the
//                column's list (atomic cursor; lists hold 3 k + 8 sigma entries);
//   4. finalize: per query, select the k best of its list, order them, translate plane rows to the caller's indices.
//                A list that overflowed or ended short of k (adversarial data: thousands of exact ties around the
//                bound) is counted in `fail`; the host then re-runs the call on the rectangle kernel.
#pragma once
#include "epilogues.cuh"

namespace wealy {

// rows of the sample: sorted positions k * n / S, k = 0 .. S - 1 (distinct for S <= n) -> their plane rows copied into
// a dense [S][d_pad] operand (hi plane only: the pre-pass runs one fp16 pass)
__global__ void __launch_bounds__(256) sample_rows_kernel(const __half* __restrict__ hi, int d_pad, int n, int n_sample,
                                                          __half* __restrict__ out) {
  const int k = (int)((blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5);
  const int lane = (int)(threadIdx.x & 31);
  if (k >= n_sample) return;
  const int srow = (int)(((long long)k * n) / n_sample);
  const uint4* src = reinterpret_cast<const uint4*>(hi + (long long)spread_plane_of(srow) * d_pad);
  uint4* dst = reinterpret_cast<uint4*>(out + (long long)k * d_pad);
  for (int v = lane; v < (d_pad >> 3); v += 32) dst[v] = __ldg(src + v);
}

// Pre-pass epilogue: the maximum of every 32-column chunk ("group") of the sample, per query row -- one FMNMX per
// element, no lists, no ids.  The m-th largest of a row's group maxima is one of the sample's similarities with at
// least m - 1 others above it, hence a LOWER bound of the sample's m-th best (and, the top few of thousands rarely
// sharing a group, nearly equal to it).
struct GroupMaxParams {
  float* gmax;   // [rows][n_groups]
  int n_groups;  // sample columns / 32
};
struct GroupMaxEpi {
  using Params = GroupMaxParams;
  static constexpr int kWarpScratchBytes = 0;
  static constexpr int kCtaScratchBytes = 0;
  struct RowState {};
  __device__ static __forceinline__ void row_begin(const Params&, RowState&, int, int, const GemmShape&, const EpiCtx&) {}
  __device__ static __forceinline__ void chunk32(const Params& p, RowState&, int row, int col0, const uint32_t (&acc)[32],
                                                 const GemmShape& sh, const EpiCtx&) {
    float m = __uint_as_float(acc[0]);
#pragma unroll
    for (int e = 1; e < 32; ++e) m = fmaxf(m, __uint_as_float(acc[e]));
    if (row < sh.m_rows && col0 < sh.n_cols) p.gmax[(long long)row * p.n_groups + (col0 >> 5)] = m;
  }
  __device__ static __forceinline__ void tile_begin(const Params&, RowState&, const GemmShape&, const EpiCtx&, int) {}
  __device__ static __forceinline__ void tile_end(const Params&, RowState&, const GemmShape&, const EpiCtx&) {}
  __device__ static __forceinline__ void row_end(const Params&, RowState&, int, int, const GemmShape&, const EpiCtx&) {}
};

// beta[p] = the m-th largest group maximum of plane row p (m = r + 1: the query itself may sit in the sample with
// similarity 1 and is simply skipped over), also written into lvl[p].w where the sweep's per-tile column slots pick it
// up; padded rows keep +inf.  n_groups <= 1024.
__global__ void __launch_bounds__(128) topk_beta_kernel(const float* __restrict__ gmax, int n_groups, int n_rows, int m, int n,
                                                        float* __restrict__ beta, float4* __restrict__ lvl, int n_lvl,
                                                        int* __restrict__ tk_cnt) {
  __shared__ float sv_all[4][1024];
  __shared__ int si_all[4][1024];
  const int p = (int)((blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5);
  const int lane = (int)(threadIdx.x & 31);
  if (p >= n_lvl) return;
  float* sv = sv_all[threadIdx.x >> 5];
  int* si = si_all[threadIdx.x >> 5];
  if (lane == 0 && p < n_rows) tk_cnt[p] = 0;
  float b = __int_as_float(0x7f800000);
  if (p < n_rows && spread_sorted_of(p) < n) {
    for (int e = lane; e < n_groups; e += 32) {
      sv[e] = gmax[(long long)p * n_groups + e];
      si[e] = e;
    }
    __syncwarp();
    // (instantiated for the number of groups: 128 at the minimum sample of 4096 rows -- 4 keys per lane, not 32)
    if (n_groups <= m) b = __int_as_float(0xff800000);
    else if (n_groups <= 128) b = warp_select_topk<4>(sv, si, n_groups, m, lane);
    else if (n_groups <= 256) b = warp_select_topk<8>(sv, si, n_groups, m, lane);
    else if (n_groups <= 512) b = warp_select_topk<16>(sv, si, n_groups, m, lane);
    else b = warp_select_topk<32>(sv, si, n_groups, m, lane);
  }
  if (lane == 0) {
    if (p < n_rows) beta[p] = b;
    lvl[p].w = b;
  }
}

// k best of a list of n <= 32 * kPerLane entries, moved to its front (warp_select_topk's contract, epilogues.cuh); the
// bisection over the order keys ends as soon as EXACTLY k entries lie at or above the prefix -- further bits could only
// raise the threshold inside the gap below the k-th best, the selected set is already final (16-22 of the 32 steps on
// similarity data).
template <int kPerLane>
__device__ __noinline__ void select_topk_exact(float* val, int* idx, int n, int k, int lane) {
  constexpr unsigned kFull = 0xffffffffu;
  __syncwarp();
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
    if (c == k) break;
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
}

// The min(k, m) best of a list of m <= cap entries (plane rows) moved to its front, their plane rows translated to the
// caller's indices (the selection itself never looks at indices, so that equal similarities are ordered like the
// rectangle path orders them).  Returns min(k, m).
__device__ __forceinline__ int sym_list_best(float* sv, int* si, int m, int k, const int* __restrict__ perm, int lane) {
  // (lists are sized mean + 8 sigma: most hold far fewer entries than `cap`, so the selection is instantiated for the
  //  list's length, and its bisection stops at the first prefix that exactly k entries reach)
  if (m > k) {
    if (m <= 256) select_topk_exact<8>(sv, si, m, k, lane);
    else if (m <= 512) select_topk_exact<16>(sv, si, m, k, lane);
    else if (m <= 768) select_topk_exact<24>(sv, si, m, k, lane);
    else select_topk_exact<32>(sv, si, m, k, lane);
  }
  const int kk = m < k ? m : k;
  __syncwarp();
  for (int e = lane; e < kk; e += 32) si[e] = perm[spread_sorted_of(si[e])];
  __syncwarp();
  return kk;
}

// position of entry e among the kk entries of a list in the output order: descending similarity, ties -> lower caller
// index (like a stable ascending-distance argsort)
__device__ __forceinline__ int sym_list_rank(const float* sv, const int* si, int kk, int e) {
  const float ve = sv[e];
  const int ie = si[e];
  int r = 0;
  for (int f = 0; f < kk; ++f) {
    const float vf = sv[f];
    r += (vf > ve) || (vf == ve && si[f] < ie);
  }
  return r;
}

// finalize: one warp per plane row (query).  Its list holds every candidate above beta (plane rows); select the k best,
// order them and write them at the caller's row.  Lists that overflowed or hold fewer than k entries are reported in
// `fail`.
__global__ void __launch_bounds__(128) topk_sym_finalize_kernel(float* __restrict__ tk_val, int* __restrict__ tk_idx,
                                                                const int* __restrict__ tk_cnt, int cap, int n_rows, int n,
                                                                int k, const int* __restrict__ perm,
                                                                long long* __restrict__ out_idx, float* __restrict__ out_sim,
                                                                int* __restrict__ fail) {
  const int p = (int)((blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5);
  const int lane = (int)(threadIdx.x & 31);
  if (p >= n_rows) return;
  const int srow = spread_sorted_of(p);
  if (srow >= n) return;
  const long long q = perm[srow];
  const int m = tk_cnt[p];
  if (m > cap || m < k) {
    if (lane == 0) atomicAdd(fail, 1);
    return;
  }
  float* sv = tk_val + (long long)p * cap;
  int* si = tk_idx + (long long)p * cap;
  sym_list_best(sv, si, m, k, perm, lane);
  for (int e = lane; e < k; e += 32) {
    const int r = sym_list_rank(sv, si, k, e);
    out_idx[q * k + r] = si[e];
    out_sim[q * k + r] = sv[e];
  }
}

// Sharded sweep (wealy_eval_sweep_shard_topk): the local finalize.  A rank's list of query q holds the candidates above
// beta_q that ITS row blocks found; the min(k, m) best of it go to the caller's row q in the order above, padded with
// (-inf, -1), and cnt[q] = m (-1: the list overflowed).  A list shorter than k is no failure here -- the other ranks hold
// the rest; topk_merge_kernel judges the union.
__global__ void __launch_bounds__(128) topk_sym_local_kernel(float* __restrict__ tk_val, int* __restrict__ tk_idx,
                                                             const int* __restrict__ tk_cnt, int cap, int n_rows, int n, int k,
                                                             const int* __restrict__ perm, float* __restrict__ out_val,
                                                             int* __restrict__ out_idx, int* __restrict__ out_cnt) {
  const int p = (int)((blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5);
  const int lane = (int)(threadIdx.x & 31);
  if (p >= n_rows) return;
  const int srow = spread_sorted_of(p);
  if (srow >= n) return;
  const long long q = perm[srow];
  const int m = tk_cnt[p];
  if (lane == 0) out_cnt[q] = m > cap ? -1 : m;
  float* sv = tk_val + (long long)p * cap;
  int* si = tk_idx + (long long)p * cap;
  const int kk = m > cap ? 0 : sym_list_best(sv, si, m, k, perm, lane);
  for (int e = lane; e < k; e += 32) {
    if (e < kk) {
      const int r = sym_list_rank(sv, si, kk, e);
      out_idx[q * k + r] = si[e];
      out_val[q * k + r] = sv[e];
    } else {
      out_idx[q * k + e] = -1;
      out_val[q * k + e] = __int_as_float(0xff800000);
    }
  }
}

// Merge of the sharded lists (wealy_eval_topk_merge), one warp per query q: its `world` lists of k entries (val / idx
// [world][n][k], cnt [world][n]) -> the k best, by descending similarity, ties -> lower index.  Every entry becomes one
// 64-bit key {order key of the similarity, ~(index + 1)}, unique but for the (-inf, -1) padding (whose copies are
// identical), so the k largest keys -- found by a bisection like select_topk_exact's, on 64 bits -- and their order do
// not depend on the order of the lists.  Adds 1 to `fail` where a list overflowed (cnt -1) or the lists hold fewer than
// k entries together.  world * k <= 32 * kPerLane, k <= 128.
template <int kPerLane>
__global__ void __launch_bounds__(128) topk_merge_kernel(const float* __restrict__ val, const int* __restrict__ idx,
                                                         const int* __restrict__ cnt, int world, long long n, int k,
                                                         long long* __restrict__ out_idx, float* __restrict__ out_sim,
                                                         int* __restrict__ fail) {
  constexpr unsigned kFull = 0xffffffffu;
  __shared__ unsigned long long skey_all[4][128];
  const long long q = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  const int lane = (int)(threadIdx.x & 31);
  if (q >= n) return;
  unsigned long long* sk = skey_all[threadIdx.x >> 5];
  int total = 0;
  bool over = false;
  for (int w = lane; w < world; w += 32) {
    const int c = cnt[(long long)w * n + q];
    over |= c < 0;
    total += c < 0 ? 0 : c;
  }
  total = __reduce_add_sync(kFull, total);
  over = __any_sync(kFull, over);
  if (lane == 0 && (over || total < k)) atomicAdd(fail, 1);
  const int L = world * k;
  unsigned long long key[kPerLane];
#pragma unroll
  for (int j = 0; j < kPerLane; ++j) {
    const int e = j * 32 + lane;
    key[j] = 0ull;  // below every entry's key (the order key of -inf is 0x007fffff)
    if (e < L) {
      const int w = e / k;
      const long long o = ((long long)w * n + q) * k + (e - w * k);
      key[j] = ((unsigned long long)float_order_key(val[o]) << 32) | (unsigned)~(unsigned)(idx[o] + 1);
    }
  }
  unsigned long long T = 0ull;
  for (int b = 63; b >= 0; --b) {
    const unsigned long long cand = T | (1ull << b);
    int c = 0;
#pragma unroll
    for (int j = 0; j < kPerLane; ++j) c += key[j] >= cand;
    c = __reduce_add_sync(kFull, c);
    if (c >= k) T = cand;  // warp-uniform
    if (c == k) break;
  }
  int g = 0, e_q = 0;
#pragma unroll
  for (int j = 0; j < kPerLane; ++j) {
    g += key[j] > T;
    e_q += key[j] == T;
  }
  int gi = g, qi = e_q;  // inclusive scans over lanes
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int tg = __shfl_up_sync(kFull, gi, o);
    const int tq = __shfl_up_sync(kFull, qi, o);
    if (lane >= o) { gi += tg; qi += tq; }
  }
  int pg = gi - g;
  int pq = __shfl_sync(kFull, gi, 31) + (qi - e_q);
#pragma unroll
  for (int j = 0; j < kPerLane; ++j) {
    if (key[j] > T) sk[pg++] = key[j];
    else if (key[j] == T) {
      if (pq < k) sk[pq] = key[j];
      ++pq;
    }
  }
  __syncwarp();
  for (int e = lane; e < k; e += 32) {
    const unsigned long long ke = sk[e];
    int r = 0;
    for (int f = 0; f < k; ++f) {
      const unsigned long long kf = sk[f];
      r += (kf > ke) || (kf == ke && f < e);
    }
    out_idx[q * k + r] = (long long)(int)(~(unsigned)ke) - 1;
    out_sim[q * k + r] = float_from_order_key((unsigned)(ke >> 32));
  }
}

}  // namespace wealy
