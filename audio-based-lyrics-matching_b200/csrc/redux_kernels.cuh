// a4: distance_tensor_redux (lib/tensor_ops.py:288-373) as ONE kernel.
//
// dist (b1, b2, s1, s2) -> (b1, b2): every (query track, candidate track) pair owns an s1 x s2 block of chunk-level
// distances (s <= 32: WEALY yields a handful of chunks per track) and reduces it with one of the reference's
// strategies.  One warp per pair; the block (and its mask) is staged in shared memory, row / column aggregates are
// computed one row or column per lane.  The reference composes every strategy from full-tensor passes (masked min /
// mean, topk, a Python loop of n rounds for the greedy pairing); here the 4-D tensor is read once.
//
// Semantics follow the reference to the letter, quirks included (see oracle/masked.py, pinned by tests/golden/redux.npz):
//   * mask != 0 means EXCLUDED; excluded entries count as +-inf_ = +-1e12 in min / max, as 0 * x in sums;
//   * means divide by max(count, eps);  "meanmin" weights a row's minimum by the row's number of included entries
//     (the reference broadcasts the row minima against the full mask);  a fully excluded row drops out of "minmean";
//   * "best-k": mean of those of the k smallest values that are below inf_;  "worst-k": the reference masks out
//     everything >= -inf_, i.e. everything -> 0 (NaN / inf propagate through 0 * x);
//   * "bpwr-n": greedy best pairs without replacement on the (already jittered) block, transposed first when
//     s2 < s1; n rounds, after each of the first n - 1 every row and column whose minimum is <= the round's minimum
//     is excluded; the result is the mean of the picked entries;
//   * the "s" prefix averages the strategy on the block and on its transpose.
#pragma once
#include "prep.cuh"
#include "loss_kernels.cuh"

namespace wealy {

enum ReduxOp : int { kRdxMin = 0, kRdxMax = 1, kRdxMean = 2, kRdxMinMean = 3, kRdxMeanMin = 4, kRdxBest = 5, kRdxWorst = 6, kRdxBpwr = 7 };

constexpr int kReduxMaxS = 32;  // chunks per track on either side

// One strategy on the block held in shared memory: x[i * ld_i + j * ld_j] (i < n1 rows, j < n2 columns), mk likewise.
// kGrad: the backward reuses the forward's selection and adds scale * w_e (out = sum_e w_e x_e) to wt[i * ld_i + j * ld_j]
// for the entries it selected; the forward's arithmetic is the same in both instantiations.
template <typename A, bool kGrad = false>
__device__ A redux_block(int op, int karg, const A* x, unsigned char* mk, int n1, int n2, int ld_i, int ld_j, A eps, A inf_, int lane,
                         A* agg /*[32]*/, A* work /*[1024]*/, A* wt = nullptr, A scale = 0) {
  constexpr unsigned kFull = 0xffffffffu;
  const int n = n1 * n2;
  auto at = [&](int i, int j) { return x[i * ld_i + j * ld_j]; };
  auto ex = [&](int i, int j) { return mk[i * ld_i + j * ld_j] != 0; };
  auto wsum = [&](A v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
  };
  auto wmin = [&](A v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const A w = __shfl_xor_sync(kFull, v, o);
      v = (w < v || w != w) ? w : v;  // NaN wins, like torch.min
    }
    return v;
  };
  auto wmax = [&](A v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const A w = __shfl_xor_sync(kFull, v, o);
      v = (w > v || w != w) ? w : v;
    }
    return v;
  };
  auto same = [](A a, A b) { return a == b || (a != a && b != b); };
  auto add_w = [&](int i, int j, A v) { wt[i * ld_i + j * ld_j] += v; };
  if (op == kRdxMin || op == kRdxMax) {
    A v = op == kRdxMin ? inf_ : -inf_;
    bool any = false;
    for (int e = lane; e < n; e += 32) {
      const int i = e / n2, j = e - i * n2;
      const A w = ex(i, j) ? (op == kRdxMin ? inf_ : -inf_) : at(i, j);
      if (w != w) { v = w; any = true; }
      else if (!any) v = op == kRdxMin ? (w < v ? w : v) : (w > v ? w : v);
    }
    v = op == kRdxMin ? wmin(v) : wmax(v);
    if constexpr (kGrad) {
      // one-hot on the first extreme in row-major order of the (oriented) block, dropped when it is excluded
      int first = n;
      for (int e = lane; e < n && first == n; e += 32) {
        const int i = e / n2, j = e - i * n2;
        if (same(ex(i, j) ? (op == kRdxMin ? inf_ : -inf_) : at(i, j), v)) first = e;
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) first = min(first, __shfl_xor_sync(kFull, first, o));
      if (lane == 0 && first < n && !ex(first / n2, first % n2)) add_w(first / n2, first % n2, scale);
    }
    return v;
  }
  if (op == kRdxMean) {
    A s = 0, c = 0;
    for (int e = lane; e < n; e += 32) {
      const int i = e / n2, j = e - i * n2;
      const bool m = ex(i, j);
      s += m ? (A)0 * at(i, j) : at(i, j);
      c += m ? (A)0 : (A)1;
    }
    s = wsum(s);
    c = wsum(c);
    if constexpr (kGrad) {
      const A q = scale / (c > eps ? c : eps);
      for (int e = lane; e < n; e += 32) {
        const int i = e / n2, j = e - i * n2;
        if (!ex(i, j)) add_w(i, j, q);
      }
    }
    return s / (c > eps ? c : eps);
  }
  if (op == kRdxMinMean || op == kRdxMeanMin) {
    // one row per lane: its masked mean / masked minimum and its number of included entries
    A r = 0, cnt = 0;
    if (lane < n1) {
      if (op == kRdxMinMean) {
        A s = 0;
        for (int j = 0; j < n2; ++j) {
          const bool m = ex(lane, j);
          s += m ? (A)0 * at(lane, j) : at(lane, j);
          cnt += m ? (A)0 : (A)1;
        }
        r = s / (cnt > eps ? cnt : eps);
      } else {
        r = inf_;
        bool nan = false;
        for (int j = 0; j < n2; ++j) {
          const bool m = ex(lane, j);
          const A w = m ? inf_ : at(lane, j);
          if (w != w) { r = w; nan = true; }
          else if (!nan && w < r) r = w;
          cnt += m ? (A)0 : (A)1;
        }
      }
    }
    if (op == kRdxMinMean) {
      // min over the rows that have an included entry (their mean stands at every included position)
      A v = (lane < n1 && cnt > 0) ? r : inf_;
      v = wmin(v);
      if constexpr (kGrad) {
        // the first row with an included entry whose mean is the minimum: 1 / max(cnt_i, eps) on its included entries
        const unsigned rows = __ballot_sync(kFull, lane < n1 && cnt > 0 && same(r, v));
        if (rows) {
          const int i = __ffs(rows) - 1;
          const A ci = __shfl_sync(kFull, cnt, i);
          const A q = scale / (ci > eps ? ci : eps);
          if (lane < n2 && !ex(i, lane)) add_w(i, lane, q);
        }
      }
      return v;
    }
    // mean of the row minima, every row weighted by its number of included entries
    A s = lane < n1 ? (cnt > 0 ? cnt * r : (A)0 * r) : (A)0;
    if (lane < n1 && cnt > 0 && cnt != (A)n2) {
      // (the reference adds included * r entry by entry: same value, kept as a product)
    }
    s = wsum(s);
    const A c = wsum(lane < n1 ? cnt : (A)0);
    if constexpr (kGrad) {
      // the reference broadcasts the row minima against the mask: row i's first argmin carries cnt_i / max(C, eps)
      if (lane < n1 && cnt > 0) {
        int j = 0;
        while (j < n2 && !same(ex(lane, j) ? inf_ : at(lane, j), r)) ++j;
        if (j < n2 && !ex(lane, j)) add_w(lane, j, scale * cnt / (c > eps ? c : eps));
      }
    }
    return s / (c > eps ? c : eps);
  }
  if (op == kRdxBest || op == kRdxWorst) {
    // k smallest (largest) of the flattened block with excluded entries at +inf_ (-inf_): rank counting, n <= 1024
    const int k = karg < 1 ? 1 : (karg > n ? n : karg);
    for (int e = lane; e < n; e += 32) {
      const int i = e / n2, j = e - i * n2;
      work[e] = ex(i, j) ? (op == kRdxBest ? inf_ : -inf_) : at(i, j);
    }
    __syncwarp();
    A s = 0, c = 0;
    unsigned kept = 0;  // (kGrad) bit e / 32: this lane's entry e was selected and is included
    for (int e = lane; e < n; e += 32) {
      const A v = work[e];
      int rank = 0;
      for (int f = 0; f < n; ++f) {
        const A w = work[f];
        rank += op == kRdxBest ? ((w < v) || (w == v && f < e)) : ((w > v) || (w == v && f < e));
      }
      if (rank < k) {
        // mmean(sel, mask = sel >= ctt): best keeps what lies below +inf_, worst excludes everything (>= -inf_ always)
        const bool excluded = op == kRdxBest ? (v >= inf_) : (v >= -inf_);
        s += excluded ? (A)0 * v : v;
        c += excluded ? (A)0 : (A)1;
        if constexpr (kGrad) kept |= excluded ? 0u : 1u << (e >> 5);
      }
    }
    __syncwarp();
    s = wsum(s);
    c = wsum(c);
    if constexpr (kGrad) {
      const A q = scale / (c > eps ? c : eps);
      for (int e = lane; e < n; e += 32)
        if ((kept >> (e >> 5)) & 1u) add_w(e / n2, e - (e / n2) * n2, q);
    }
    return s / (c > eps ? c : eps);
  }
  // ---- bpwr: greedy best pairs without replacement (the block is already jittered by the caller)
  {
    const int rounds = karg < 1 ? n1 : (karg > n1 ? n1 : karg);
    unsigned char* picked = reinterpret_cast<unsigned char*>(work);  // [n] bytes inside the work area
    for (int e = lane; e < n; e += 32) picked[e] = 0;
    __syncwarp();
    for (int it = 0; it < rounds; ++it) {
      A best = inf_;
      for (int e = lane; e < n; e += 32) {
        const int i = e / n2, j = e - i * n2;
        const A w = ex(i, j) ? inf_ : at(i, j);
        best = w < best ? w : best;
      }
      best = wmin(best);
      for (int e = lane; e < n; e += 32) {
        const int i = e / n2, j = e - i * n2;
        if (!ex(i, j) && at(i, j) <= best) picked[e] = 1;
      }
      if (it < rounds - 1) {
        // rows / columns whose minimum over the included entries is <= best drop out (one row and one column per lane)
        bool row_out = false, col_out = false;
        if (lane < n1) {
          A m = inf_;
          for (int j = 0; j < n2; ++j) { const A w = ex(lane, j) ? inf_ : at(lane, j); m = w < m ? w : m; }
          row_out = m <= best;
        }
        if (lane < n2) {
          A m = inf_;
          for (int i = 0; i < n1; ++i) { const A w = ex(i, lane) ? inf_ : at(i, lane); m = w < m ? w : m; }
          col_out = m <= best;
        }
        __syncwarp();
        const unsigned rows = __ballot_sync(kFull, row_out), cols = __ballot_sync(kFull, col_out);
        for (int e = lane; e < n; e += 32) {
          const int i = e / n2, j = e - i * n2;
          if (((rows >> i) & 1u) || ((cols >> j) & 1u)) mk[i * ld_i + j * ld_j] = 1;
        }
      }
      __syncwarp();
    }
    A s = 0, c = 0;
    for (int e = lane; e < n; e += 32) {
      const int i = e / n2, j = e - i * n2;
      s += picked[e] ? at(i, j) : (A)0 * at(i, j);
      c += picked[e] ? (A)1 : (A)0;
    }
    s = wsum(s);
    c = wsum(c);
    if constexpr (kGrad) {
      const A q = scale / (c > eps ? c : eps);
      for (int e = lane; e < n; e += 32)
        if (picked[e]) add_w(e / n2, e - (e / n2) * n2, q);
    }
    (void)agg;
    return s / (c > eps ? c : eps);
  }
}

template <typename A>
__host__ __device__ constexpr int redux_warps() { return sizeof(A) == 8 ? 2 : 4; }  // static shared memory: 2 x 1024 A + 2 x 1024 bytes per warp

// The strategy on one staged block (xs, ms = working mask, ms0 = the caller's mask), "s" prefix included.  bpwr works on
// the orientation with the fewer rows (the reference transposes when s2 < s1).  kGrad: the weights go to wt (zeroed).
template <typename A, bool kGrad = false>
__device__ __forceinline__ A redux_pair(int op, int karg, int symmetric, const A* xs, unsigned char* ms, const unsigned char* ms0,
                                        int s1, int s2, A eps, A inf_, int lane, A* ag, A* ws, A* wt = nullptr) {
  const int n = s1 * s2;
  const bool bp = op == kRdxBpwr;
  const A scale = symmetric ? (A)0.5 : (A)1;
  auto run = [&](bool transposed) {
    const bool t = transposed != (bp && ((transposed ? s1 : s2) < (transposed ? s2 : s1)));
    const int n1 = t ? s2 : s1, n2 = t ? s1 : s2;
    return redux_block<A, kGrad>(op, karg, xs, ms, n1, n2, t ? 1 : s2, t ? s2 : 1, eps, inf_, lane, ag, ws, wt, scale);
  };
  A r = run(false);
  if (symmetric) {
    __syncwarp();
    for (int e = lane; e < n; e += 32) ms[e] = ms0[e];  // (bpwr edits its mask)
    __syncwarp();
    r = (A)0.5 * (r + run(true));
  }
  return r;
}

template <typename T, typename A>
__global__ void __launch_bounds__(128) redux_pairs_kernel(const T* __restrict__ dist, const unsigned char* __restrict__ mask,
                                                          long long pairs, int s1, int s2, int op, int karg, int symmetric, A eps,
                                                          A inf_, T* __restrict__ out) {
  constexpr int kW = redux_warps<A>();
  __shared__ A xs[kW][kReduxMaxS * kReduxMaxS];
  __shared__ A ws[kW][kReduxMaxS * kReduxMaxS];
  __shared__ unsigned char ms[kW][kReduxMaxS * kReduxMaxS];
  __shared__ unsigned char ms0[kW][kReduxMaxS * kReduxMaxS];
  __shared__ A ag[kW][32];
  const int w = (int)(threadIdx.x >> 5), lane = (int)(threadIdx.x & 31);
  const long long pair = blockIdx.x * (long long)kW + w;
  if (pair >= pairs) return;
  const int n = s1 * s2;
  const T* src = dist + pair * n;
  for (int e = lane; e < n; e += 32) {
    if constexpr (sizeof(A) == 8) xs[w][e] = (A)src[e]; else xs[w][e] = (A)to_f32<T>(src[e]);
    ms0[w][e] = mask ? (unsigned char)(mask[pair * n + e] != 0) : 0;
    ms[w][e] = ms0[w][e];
  }
  __syncwarp();
  const A r = redux_pair<A>(op, karg, symmetric, xs[w], ms[w], ms0[w], s1, s2, eps, inf_, lane, ag[w], ws[w]);
  if (lane == 0) {
    if constexpr (sizeof(A) == 8) out[pair] = (T)r; else out[pair] = from_f32<T>((float)r);
  }
}

// The backward of one track pair: d dist[pair][e] = g[pair] * w_e, w_e written by the forward's selection (redux_block<A, true>)
// rerun on the same (jittered, for bpwr) block.  One warp per pair like the forward; the weights take a third block of
// shared memory, so a CTA holds one warp fewer (float) / one warp (double) to stay within the 48 KB of static shared memory.
template <typename A>
__host__ __device__ constexpr int redux_bwd_warps() { return sizeof(A) == 8 ? 1 : 3; }

template <typename T, typename A>
__global__ void __launch_bounds__(96) redux_pairs_backward_kernel(const T* __restrict__ dist, const unsigned char* __restrict__ mask,
                                                                  long long pairs, int s1, int s2, int op, int karg, int symmetric,
                                                                  A eps, A inf_, const T* __restrict__ g, T* __restrict__ dx) {
  constexpr int kW = redux_bwd_warps<A>();
  __shared__ A xs[kW][kReduxMaxS * kReduxMaxS];
  __shared__ A ws[kW][kReduxMaxS * kReduxMaxS];
  __shared__ A wt[kW][kReduxMaxS * kReduxMaxS];
  __shared__ unsigned char ms[kW][kReduxMaxS * kReduxMaxS];
  __shared__ unsigned char ms0[kW][kReduxMaxS * kReduxMaxS];
  __shared__ A ag[kW][32];
  const int w = (int)(threadIdx.x >> 5), lane = (int)(threadIdx.x & 31);
  const long long pair = blockIdx.x * (long long)kW + w;
  if (pair >= pairs) return;
  const int n = s1 * s2;
  const T* src = dist + pair * n;
  for (int e = lane; e < n; e += 32) {
    if constexpr (sizeof(A) == 8) xs[w][e] = (A)src[e]; else xs[w][e] = (A)to_f32<T>(src[e]);
    ms0[w][e] = mask ? (unsigned char)(mask[pair * n + e] != 0) : 0;
    ms[w][e] = ms0[w][e];
    wt[w][e] = 0;
  }
  __syncwarp();
  redux_pair<A, true>(op, karg, symmetric, xs[w], ms[w], ms0[w], s1, s2, eps, inf_, lane, ag[w], ws[w], wt[w]);
  __syncwarp();
  A gp;
  if constexpr (sizeof(A) == 8) gp = (A)g[pair]; else gp = (A)to_f32<T>(g[pair]);
  T* d = dx + pair * n;
  for (int e = lane; e < n; e += 32) {
    if constexpr (sizeof(A) == 8) d[e] = (T)(gp * wt[w][e]); else d[e] = from_f32<T>((float)(gp * wt[w][e]));
  }
}

}  // namespace wealy
