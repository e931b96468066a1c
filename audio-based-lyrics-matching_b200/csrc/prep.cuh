// K0 `prep_rows`: one HBM pass over the embeddings that
//   * computes the row L2 norm (and squared norm, max |x|),
//   * applies the reference's normalisation  x / (|x| + eps)   [lib/tensor_ops.py:169-170]
//     or F.normalize's  x / max(|x|, eps)                       [lib/losses.py:231]
//     or, for dot / euclidean modes, an exact power-of-two row scaling (folded back in the epilogue),
//   * splits the result into the fp16 `hi` plane and the fp16 residual `lo` plane the
//     tensor-core contraction consumes (x ~= hi + lo to ~2^-22), zero-padding K to the k-block,
//   * optionally accumulates the logdict statistics (max |z|, sum z, sum z^2; lib/losses.py:69-71,281-283).
// HBM-bound: reads n*d*sizeof(T), writes n*d_pad*2*planes bytes.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "ptx.cuh"

namespace wealy {

enum PrepMode : int {
  kPrepL2AddEps = 0,  // x / (|x| + eps)
  kPrepL2Clamp = 1,   // x / max(|x|, eps)
  kPrepRawPow2 = 2,   // x * 2^-e, e = exponent of max|x|; epilogue multiplies by 2^e
};

// Statistics of z for the losses' logdict.  Every warp adds its row's share with atomics; 32 slots (picked by block
// index) keep thousands of same-address atomics from serialising on one L2 line -- the reader sums the slots.
constexpr int kZSlots = 32;
struct ZStats {
  double sum[kZSlots];
  double sumsq[kZSlots];
  unsigned int maxabs_bits[kZSlots];  // float bits of max |z| (non-negative floats order like uints)
};

template <typename T>
__device__ __forceinline__ float to_f32(T v);
template <>
__device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <>
__device__ __forceinline__ float to_f32<__half>(__half v) { return __half2float(v); }
template <>
__device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }

// four consecutive elements as floats (16-bit types: one 8-byte access, fp32: one 16-byte access)
template <typename T>
__device__ __forceinline__ float4 load4(const T* p);
template <>
__device__ __forceinline__ float4 load4<float>(const float* p) { return *reinterpret_cast<const float4*>(p); }
template <>
__device__ __forceinline__ float4 load4<__half>(const __half* p) {
  const uint2 v = *reinterpret_cast<const uint2*>(p);
  const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&v.x)), b = __half22float2(*reinterpret_cast<const __half2*>(&v.y));
  return make_float4(a.x, a.y, b.x, b.y);
}
template <>
__device__ __forceinline__ float4 load4<__nv_bfloat16>(const __nv_bfloat16* p) {
  const uint2 v = *reinterpret_cast<const uint2*>(p);
  const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&v.x)),
               b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&v.y));
  return make_float4(a.x, a.y, b.x, b.y);
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// One warp per row.  `hi_t` / `lo_t` (optional) receive the transposed planes [d_pad_t rows = d][n_pad_t]
// used as the K-major "B" operand of the  dU = W * U  product of the loss backward.
template <typename T>
__global__ void __launch_bounds__(256) prep_rows_kernel(const T* __restrict__ x, long long ld, int n, int d, int d_pad,
                                                        int mode, float eps, int stats_on_scaled,
                                                        __half* __restrict__ hi, __half* __restrict__ lo,
                                                        __half* __restrict__ hi_t, __half* __restrict__ lo_t,
                                                        long long ld_t, float* __restrict__ norm_out,
                                                        float* __restrict__ scale_out, float* __restrict__ sq_out,
                                                        ZStats* __restrict__ stats,
                                                        const int* __restrict__ gather = nullptr, int spread_n = 0) {
  const int warp = (int)((blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5);
  const int lane = (int)(threadIdx.x & 31);
  if (warp >= n) return;
  // `gather` (optional): output row r is built from input row gather[r] (clique-sorted planes of the evaluation sweep);
  // spread_n > 0: the n output rows are in the sweep's spread order (gemm_core.cuh) over spread_n sorted rows --
  // output row r holds sorted row spread_sorted_of(r), rows past the end are zero
  int src = warp;
  if (spread_n > 0) {
    src = (warp & ~127) + (((warp & 127) & 31) << 2) + ((warp & 127) >> 5);
    if (src >= spread_n) {
      for (int k = lane; k < d_pad; k += 32) {
        hi[(long long)warp * d_pad + k] = __float2half_rn(0.f);
        if (lo) lo[(long long)warp * d_pad + k] = __float2half_rn(0.f);
      }
      if (lane == 0) {
        if (norm_out) norm_out[warp] = 0.f;
        if (scale_out) scale_out[warp] = 1.f;
        if (sq_out) sq_out[warp] = 0.f;
      }
      return;
    }
  }
  const T* row = x + (long long)(gather ? gather[src] : src) * ld;

  // HBM-bound row passes: 4 elements per lane and access when the rows are suitably aligned (the usual case)
  const bool vec = (d % 4 == 0) && (ld % 4 == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0) && hi_t == nullptr;
  float ss = 0.f, mx = 0.f;
  if (vec) {
    for (int k = lane * 4; k < d; k += 128) {
      const float4 v = load4<T>(row + k);
      ss = fmaf(v.x, v.x, ss); ss = fmaf(v.y, v.y, ss); ss = fmaf(v.z, v.z, ss); ss = fmaf(v.w, v.w, ss);
      mx = fmaxf(fmaxf(mx, fmaxf(fabsf(v.x), fabsf(v.y))), fmaxf(fabsf(v.z), fabsf(v.w)));
    }
  } else {
    for (int k = lane; k < d; k += 32) {
      const float v = to_f32<T>(row[k]);
      ss = fmaf(v, v, ss);
      mx = fmaxf(mx, fabsf(v));
    }
  }
  ss = warp_sum(ss);
  mx = warp_max(mx);
  const float nrm = sqrtf(ss);

  float div = 1.f;   // x_hat = x / div
  float escale = 1.f;  // epilogue row factor
  if (mode == kPrepL2AddEps) {
    div = nrm + eps;
  } else if (mode == kPrepL2Clamp) {
    div = fmaxf(nrm, eps);
  } else {
    int e = 0;
    if (mx > 0.f) frexpf(mx, &e);  // mx = f * 2^e, f in [0.5, 1)  ->  |x * 2^-e| < 1
    div = ldexpf(1.f, e);
    escale = div;
  }

  double s1 = 0.0, s2 = 0.0;
  float smx = 0.f;
  __half* hrow = hi + (long long)warp * d_pad;
  __half* lrow = lo ? lo + (long long)warp * d_pad : nullptr;
  if (vec) {
    for (int k = lane * 4; k < d_pad; k += 128) {  // d_pad is a multiple of 64, d of 4: a group is all data or all padding
      float4 r = make_float4(0.f, 0.f, 0.f, 0.f), v = r;
      if (k < d) {
        r = load4<T>(row + k);
        v = make_float4(r.x / div, r.y / div, r.z / div, r.w / div);  // IEEE division, as torch does
      }
      const __half2 h0 = __floats2half2_rn(v.x, v.y), h1 = __floats2half2_rn(v.z, v.w);
      uint2 oh;
      oh.x = *reinterpret_cast<const unsigned*>(&h0);
      oh.y = *reinterpret_cast<const unsigned*>(&h1);
      *reinterpret_cast<uint2*>(hrow + k) = oh;
      if (lrow) {
        const float2 f0 = __half22float2(h0), f1 = __half22float2(h1);
        const __half2 l0 = __floats2half2_rn(v.x - f0.x, v.y - f0.y), l1 = __floats2half2_rn(v.z - f1.x, v.w - f1.y);
        uint2 ol;
        ol.x = *reinterpret_cast<const unsigned*>(&l0);
        ol.y = *reinterpret_cast<const unsigned*>(&l1);
        *reinterpret_cast<uint2*>(lrow + k) = ol;
      }
      if (stats && k < d) {
        const float4 sv = stats_on_scaled ? v : r;
        s1 += (double)sv.x + (double)sv.y + (double)sv.z + (double)sv.w;
        s2 += (double)sv.x * sv.x + (double)sv.y * sv.y + (double)sv.z * sv.z + (double)sv.w * sv.w;
        smx = fmaxf(fmaxf(smx, fmaxf(fabsf(sv.x), fabsf(sv.y))), fmaxf(fabsf(sv.z), fabsf(sv.w)));
      }
    }
  } else {
  for (int k = lane; k < d_pad; k += 32) {
    float v = 0.f;
    if (k < d) v = to_f32<T>(row[k]) / div;  // IEEE division, as torch does
    const __half h = __float2half_rn(v);
    hrow[k] = h;
    __half l = __float2half_rn(0.f);
    if (lrow) {
      l = __float2half_rn(v - __half2float(h));
      lrow[k] = l;
    }
    if (hi_t && k < d) {
      hi_t[(long long)k * ld_t + warp] = h;
      if (lo_t) lo_t[(long long)k * ld_t + warp] = l;
    }
    if (stats && k < d) {
      const float sv = stats_on_scaled ? v : to_f32<T>(row[k]);
      s1 += (double)sv;
      s2 += (double)sv * (double)sv;
      smx = fmaxf(smx, fabsf(sv));
    }
  }
  }
  if (lane == 0) {
    if (norm_out) norm_out[warp] = nrm;
    if (scale_out) scale_out[warp] = escale;
    if (sq_out) sq_out[warp] = ss;
  }
  if (stats) {
    s1 = warp_sum_d(s1);
    s2 = warp_sum_d(s2);
    smx = warp_max(smx);
    if (lane == 0) {
      const int slot = (int)((blockIdx.x * 8u + (threadIdx.x >> 5)) % kZSlots);
      atomicAdd(&stats->sum[slot], s1);
      atomicAdd(&stats->sumsq[slot], s2);
      atomicMax(&stats->maxabs_bits[slot], __float_as_uint(smx));
    }
  }
}

// K0 for embeddings that still live in PINNED HOST memory (wealy_eval_run_host): the same arithmetic as
// prep_rows_kernel (identical summation order, IEEE division -> bit-identical planes), but every input row is read
// exactly ONCE -- it crosses PCIe -- and kept in registers between the norm and the split.  A small persistent grid,
// rows dealt warp by warp: 8 CTAs of kThreads = 512 on SMs of their own (api.cu: host_upload_setup), so that the
// upload of the next rows runs while the tensor cores of the other SMs sweep the rows that have arrived (upload warps
// NEXT TO the sweep's CTAs were measured slower: api.cu, kHostUpSms).
// Plane rows [row_lo, row_hi), whole 128-row blocks of the spread order; d <= 128 kRowVecs.
constexpr int kRowVecs = 8;  // float4 per lane: rows of up to 1024 elements
template <typename T, int kThreads>
__global__ void __launch_bounds__(kThreads) prep_rows_stream_kernel(const T* __restrict__ x, long long ld, int row_lo, int row_hi,
                                                              int d, int d_pad, float eps, __half* __restrict__ hi,
                                                              __half* __restrict__ lo, float* __restrict__ norm_out,
                                                              float* __restrict__ scale_out, float* __restrict__ sq_out,
                                                              const int* __restrict__ gather, int spread_n) {
  const int lane = (int)(threadIdx.x & 31);
  const int n_warps = (int)(gridDim.x * (blockDim.x >> 5));
  for (int r = row_lo + (int)(blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)); r < row_hi; r += n_warps) {
    const int src = (r & ~127) + (((r & 127) & 31) << 2) + ((r & 127) >> 5);  // sorted row of plane row r
    __half* hrow = hi + (long long)r * d_pad;
    __half* lrow = lo ? lo + (long long)r * d_pad : nullptr;
    if (src >= spread_n) {  // padding up to the whole block: zero rows
      for (int k = lane * 4; k < d_pad; k += 128) {
        *reinterpret_cast<uint2*>(hrow + k) = make_uint2(0u, 0u);
        if (lrow) *reinterpret_cast<uint2*>(lrow + k) = make_uint2(0u, 0u);
      }
      if (lane == 0) {
        if (norm_out) norm_out[r] = 0.f;
        if (scale_out) scale_out[r] = 1.f;
        if (sq_out) sq_out[r] = 0.f;
      }
      continue;
    }
    const T* row = x + (long long)__ldg(gather + src) * ld;
    float4 v[kRowVecs];
#pragma unroll
    for (int i = 0; i < kRowVecs; ++i) {  // all of the row's loads in flight together
      const int k = lane * 4 + i * 128;
      v[i] = k < d ? load4<T>(row + k) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    float ss = 0.f;
#pragma unroll
    for (int i = 0; i < kRowVecs; ++i) {
      if (lane * 4 + i * 128 < d) {
        ss = fmaf(v[i].x, v[i].x, ss); ss = fmaf(v[i].y, v[i].y, ss); ss = fmaf(v[i].z, v[i].z, ss); ss = fmaf(v[i].w, v[i].w, ss);
      }
    }
    ss = warp_sum(ss);
    const float nrm = sqrtf(ss);
    const float div = nrm + eps;
#pragma unroll
    for (int i = 0; i < kRowVecs; ++i) {
      const int k = lane * 4 + i * 128;
      if (k < d_pad) {
        float4 q = make_float4(0.f, 0.f, 0.f, 0.f);
        if (k < d) q = make_float4(v[i].x / div, v[i].y / div, v[i].z / div, v[i].w / div);  // IEEE division, as torch does
        const __half2 h0 = __floats2half2_rn(q.x, q.y), h1 = __floats2half2_rn(q.z, q.w);
        uint2 oh;
        oh.x = *reinterpret_cast<const unsigned*>(&h0);
        oh.y = *reinterpret_cast<const unsigned*>(&h1);
        *reinterpret_cast<uint2*>(hrow + k) = oh;
        if (lrow) {
          const float2 f0 = __half22float2(h0), f1 = __half22float2(h1);
          const __half2 l0 = __floats2half2_rn(q.x - f0.x, q.y - f0.y), l1 = __floats2half2_rn(q.z - f1.x, q.w - f1.y);
          uint2 ol;
          ol.x = *reinterpret_cast<const unsigned*>(&l0);
          ol.y = *reinterpret_cast<const unsigned*>(&l1);
          *reinterpret_cast<uint2*>(lrow + k) = ol;
        }
      }
    }
    if (lane == 0) {
      if (norm_out) norm_out[r] = nrm;
      if (scale_out) scale_out[r] = 1.f;
      if (sq_out) sq_out[r] = ss;
    }
  }
}

}  // namespace wealy
