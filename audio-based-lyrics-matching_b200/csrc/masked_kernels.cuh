// a3: masked reductions (lib/tensor_ops.py:182-258) as one HBM-bound pass: x and the exclusion mask
// are read once (coalesced), never materialising `included * x` or the +-inf filled copy the
// reference builds.  Mask polarity: non-zero == EXCLUDED (lib/tensor_ops.py:186,201,219).
#pragma once
#include "prep.cuh"
#include "loss_kernels.cuh"

namespace wealy {

enum MaskedOp : int { kMSum = 0, kMMean = 1, kMMin = 2, kMMax = 3 };

struct MaskedAcc {
  float sum, cnt, mn, mx;
};

template <typename T>
__device__ __forceinline__ void masked_visit(MaskedAcc& a, const T* __restrict__ x, const unsigned char* __restrict__ mask,
                                             long long i, float fill) {
  const float v = to_f32<T>(x[i]);
  const bool excluded = mask != nullptr && mask[i] != 0;
  // reference arithmetic: included * x (so an excluded inf/nan still poisons the sum, as upstream)
  a.sum += excluded ? 0.f * v : v;
  a.cnt += excluded ? 0.f : 1.f;
  const float w = excluded ? fill : v;
  a.mn = fminf(a.mn, w);
  a.mx = fmaxf(a.mx, w);
  if (w != w) { a.mn = w; a.mx = w; }  // torch.min / max propagate NaN
}

__device__ __forceinline__ float masked_result(const MaskedAcc& a, int op, float eps) {
  switch (op) {
    case kMSum: return a.sum;
    case kMMean: return a.sum / fmaxf(a.cnt, eps);  // den.clamp(min=eps), lib/tensor_ops.py:212
    case kMMin: return a.mn;
    default: return a.mx;
  }
}

// one warp per row (short rows: chunk-level reductions, per-anchor statistics)
template <typename T>
__global__ void __launch_bounds__(256) masked_reduce_warp_kernel(const T* __restrict__ x,
                                                                 const unsigned char* __restrict__ mask, long long rows,
                                                                 long long cols, int op, float fill, float eps,
                                                                 T* __restrict__ out) {
  const long long row = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  const int lane = (int)(threadIdx.x & 31);
  if (row >= rows) return;
  MaskedAcc a{0.f, 0.f, __int_as_float(0x7f800000), __int_as_float(0xff800000)};
  const long long base = row * cols;
  for (long long c = lane; c < cols; c += 32) masked_visit<T>(a, x, mask, base + c, fill);
  a.sum = warp_sum(a.sum);
  a.cnt = warp_sum(a.cnt);
  const bool nan = __any_sync(0xffffffffu, a.mn != a.mn);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    a.mn = fminf(a.mn, __shfl_xor_sync(0xffffffffu, a.mn, o));
    a.mx = fmaxf(a.mx, __shfl_xor_sync(0xffffffffu, a.mx, o));
  }
  if (nan) a.mn = a.mx = __int_as_float(0x7fc00000);
  if (lane == 0) out[row] = from_f32<T>(masked_result(a, op, eps));
}

// one block per row (long rows: whole-matrix statistics such as v_dpos / v_dneg, lib/losses.py:267-268)
template <typename T>
__global__ void __launch_bounds__(1024) masked_reduce_block_kernel(const T* __restrict__ x,
                                                                   const unsigned char* __restrict__ mask, long long rows,
                                                                   long long cols, int op, float fill, float eps,
                                                                   T* __restrict__ out) {
  __shared__ float s_sum[32], s_cnt[32], s_mn[32], s_mx[32];
  __shared__ int s_nan;
  const long long row = blockIdx.x;
  if (threadIdx.x == 0) s_nan = 0;
  __syncthreads();
  MaskedAcc a{0.f, 0.f, __int_as_float(0x7f800000), __int_as_float(0xff800000)};
  const long long base = row * cols;
  for (long long c = threadIdx.x; c < cols; c += blockDim.x) masked_visit<T>(a, x, mask, base + c, fill);
  if (a.mn != a.mn) atomicOr(&s_nan, 1);
  a.sum = warp_sum(a.sum);
  a.cnt = warp_sum(a.cnt);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    a.mn = fminf(a.mn, __shfl_xor_sync(0xffffffffu, a.mn, o));
    a.mx = fmaxf(a.mx, __shfl_xor_sync(0xffffffffu, a.mx, o));
  }
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) { s_sum[w] = a.sum; s_cnt[w] = a.cnt; s_mn[w] = a.mn; s_mx[w] = a.mx; }
  __syncthreads();
  if (w == 0) {
    const int nw = blockDim.x >> 5;
    MaskedAcc b{l < nw ? s_sum[l] : 0.f, l < nw ? s_cnt[l] : 0.f, l < nw ? s_mn[l] : __int_as_float(0x7f800000),
                l < nw ? s_mx[l] : __int_as_float(0xff800000)};
    b.sum = warp_sum(b.sum);
    b.cnt = warp_sum(b.cnt);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      b.mn = fminf(b.mn, __shfl_xor_sync(0xffffffffu, b.mn, o));
      b.mx = fmaxf(b.mx, __shfl_xor_sync(0xffffffffu, b.mx, o));
    }
    if (s_nan) b.mn = b.mx = __int_as_float(0x7fc00000);
    if (l == 0) out[row] = from_f32<T>(masked_result(b, op, eps));
  }
}

// ---- backward: dx = g[row] * w_e, the weights fixed by the forward's selection (rerun here, no index output) ----
//   sum: 1 on included entries;  mean: 1 / max(count, eps) on included entries;
//   min / max over given dims: one-hot on the FIRST extreme of the filled row (excluded entries hold `fill`, a NaN is
//     the extreme), dropped when that entry is excluded -- the caller orders the columns so that "first" is the
//     reference's order (it reduces the dims one at a time with torch.min(d));
//   min / max with dim=None (full != 0): torch.min() spreads the gradient evenly over every position equal to the
//     extreme (NaN: every NaN), excluded positions included in the count, their share dropped.
// Arithmetic in A (float, double for float64 inputs); dx in x's dtype.
template <typename A, typename T>
__device__ __forceinline__ A ld_acc(const T* p, long long i) {
  if constexpr (sizeof(A) == 8) return (A)p[i]; else return (A)to_f32<T>(p[i]);
}
template <typename T, typename A>
__device__ __forceinline__ void st_acc(T* p, long long i, A v) {
  if constexpr (sizeof(A) == 8) p[i] = (T)v; else p[i] = from_f32<T>((float)v);
}

template <typename A>
__device__ __forceinline__ bool same_value(A a, A b) { return a == b || (a != a && b != b); }

// a strictly more extreme than b (a NaN beats every number)
template <typename A>
__device__ __forceinline__ bool beats(A a, A b, bool take_min) {
  if (a != a) return b == b;
  return take_min ? a < b : a > b;
}

template <typename A>
struct MaskedSel {
  A cnt;          // included entries (mean)
  A v;            // extreme of the filled row (min / max)
  long long idx;  // its first position
  long long ties; // positions equal to it
  __device__ __forceinline__ void take(A w, long long i, long long t, bool take_min) {
    if (beats(w, v, take_min)) { v = w; idx = i; ties = t; }
    else if (same_value(w, v)) { ties += t; idx = i < idx ? i : idx; }
  }
  __device__ __forceinline__ void warp_merge(bool take_min) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
      const A ov = __shfl_xor_sync(0xffffffffu, v, o);
      const long long oi = __shfl_xor_sync(0xffffffffu, idx, o), ot = __shfl_xor_sync(0xffffffffu, ties, o);
      take(ov, oi, ot, take_min);
    }
  }
};

template <typename T, typename A>
__device__ __forceinline__ void masked_sel_visit(MaskedSel<A>& s, const T* __restrict__ x, const unsigned char* __restrict__ mask,
                                                 long long base, long long c, int op, A fill) {
  const bool excluded = mask != nullptr && mask[base + c] != 0;
  if (op == kMMean) { s.cnt += excluded ? (A)0 : (A)1; return; }
  s.take(excluded ? fill : ld_acc<A>(x, base + c), c, 1, op == kMMin);
}

template <typename T, typename A>
__device__ __forceinline__ void masked_grad_write(const MaskedSel<A>& s, const T* __restrict__ x,
                                                  const unsigned char* __restrict__ mask, long long base, long long c, int op,
                                                  int full, A fill, A eps, A g, T* __restrict__ dx) {
  const bool excluded = mask != nullptr && mask[base + c] != 0;
  A d;
  if (op == kMSum) d = g * (excluded ? (A)0 : (A)1);
  else if (op == kMMean) d = (g / (s.cnt > eps ? s.cnt : eps)) * (excluded ? (A)0 : (A)1);
  else if (!full) d = (c == s.idx && !excluded) ? g : (A)0;
  else d = (!excluded && same_value(ld_acc<A>(x, base + c), s.v)) ? g / (A)s.ties : (A)0;
  st_acc<T>(dx, base + c, d);
}

template <typename A>
__device__ __forceinline__ MaskedSel<A> masked_sel_init(int op) {
  const A inf = (A)__int_as_float(0x7f800000);
  return MaskedSel<A>{(A)0, op == kMMin ? inf : -inf, 0x7fffffffffffffffll, 0};
}

// one warp per row
template <typename T, typename A>
__global__ void __launch_bounds__(256) masked_reduce_backward_warp_kernel(const T* __restrict__ x,
                                                                          const unsigned char* __restrict__ mask, long long rows,
                                                                          long long cols, int op, int full, A fill, A eps,
                                                                          const T* __restrict__ g, T* __restrict__ dx) {
  const long long row = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  const int lane = (int)(threadIdx.x & 31);
  if (row >= rows) return;
  const long long base = row * cols;
  MaskedSel<A> s = masked_sel_init<A>(op);
  if (op != kMSum) {
    for (long long c = lane; c < cols; c += 32) masked_sel_visit<T, A>(s, x, mask, base, c, op, fill);
    s.warp_merge(op == kMMin);
  }
  const A gr = ld_acc<A>(g, row);
  for (long long c = lane; c < cols; c += 32) masked_grad_write<T, A>(s, x, mask, base, c, op, full, fill, eps, gr, dx);
}

// one block per row (long rows)
template <typename T, typename A>
__global__ void __launch_bounds__(1024) masked_reduce_backward_block_kernel(const T* __restrict__ x,
                                                                            const unsigned char* __restrict__ mask, long long rows,
                                                                            long long cols, int op, int full, A fill, A eps,
                                                                            const T* __restrict__ g, T* __restrict__ dx) {
  __shared__ MaskedSel<A> s_sel[32];
  const long long row = blockIdx.x;
  const long long base = row * cols;
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  MaskedSel<A> s = masked_sel_init<A>(op);
  if (op != kMSum) {
    for (long long c = threadIdx.x; c < cols; c += blockDim.x) masked_sel_visit<T, A>(s, x, mask, base, c, op, fill);
    s.warp_merge(op == kMMin);
    if (l == 0) s_sel[w] = s;
    __syncthreads();
    if (w == 0) {
      s = l < (int)(blockDim.x >> 5) ? s_sel[l] : masked_sel_init<A>(op);
      s.warp_merge(op == kMMin);
      if (l == 0) s_sel[0] = s;
    }
    __syncthreads();
    s = s_sel[0];
  }
  const A gr = ld_acc<A>(g, row);
  for (long long c = threadIdx.x; c < cols; c += blockDim.x) masked_grad_write<T, A>(s, x, mask, base, c, op, full, fill, eps, gr, dx);
}

}  // namespace wealy
