// Small kernels around the fused evaluation sweep (all HBM / latency bound, KB-MB of data):
//   ids_to_i32       int64 ids -> int32 with range check
//   segment_lookup   per query: its clique's segment in the clique-sorted candidate order
//   pos_thresholds   K_pos: relevant similarities of every query, sorted ascending (CSR)
//   ap_reduce        K2: rank counts -> AP, R1 per query (+ running sums for MAP / MR1)
//   topk_finalize    K3: merge the per-part candidate buffers into the final top-k
#pragma once
#include <cuda_fp16.h>

#include "epilogues.cuh"
#include "prep.cuh"

namespace wealy {

__global__ void ids_to_i32_kernel(const long long* __restrict__ in, int* __restrict__ out, int n, int* bad) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const long long v = in[t];
  if (v > 2147483647ll || v < -2147483648ll) atomicAdd(bad, 1);
  out[t] = (int)v;
}

// do two (clique, version) id sets hold the same values?  (an all-vs-all call may pass equal but distinct tensors)
__global__ void ids_differ_kernel(const long long* __restrict__ a_c, const long long* __restrict__ a_i,
                                  const long long* __restrict__ b_c, const long long* __restrict__ b_i, int n, int* differ) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n && (a_c[t] != b_c[t] || a_i[t] != b_i[t])) *differ = 1;
}

__global__ void iota_kernel(int* out, int n) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) out[t] = t;
}

// sorted_c: candidate clique ids ascending; sorted_idx: candidate index at each sorted position.
// For every query: [seg_lo, seg_lo + seg_len) = candidates of its clique, npos = those whose version id
// differs from the query's (lib/losses.py:40-42: positives = same label & different idx).
__global__ void segment_lookup_kernel(const int* __restrict__ q_c, const int* __restrict__ q_i, int nq,
                                      const int* __restrict__ sorted_c, const int* __restrict__ sorted_idx,
                                      const int* __restrict__ c_i, int nc, int* __restrict__ seg_lo,
                                      int* __restrict__ seg_len, int* __restrict__ npos,
                                      unsigned long long* __restrict__ totals /*[0]=queries w/o positives,[1]=max P,[4]=max len*/) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= nq) return;
  const int key = q_c[q];
  int lo = 0, hi = nc;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (sorted_c[mid] < key) lo = mid + 1; else hi = mid;
  }
  const int first = lo;
  hi = nc;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (sorted_c[mid] <= key) lo = mid + 1; else hi = mid;
  }
  const int len = lo - first;
  const int qi = q_i[q];
  int np = 0;
  for (int m = 0; m < len; ++m) np += (c_i[sorted_idx[first + m]] != qi);
  seg_lo[q] = first;
  seg_len[q] = len;
  npos[q] = np;
  if (np == 0) atomicAdd(&totals[0], 1ull);
  atomicMax(&totals[1], (unsigned long long)np);
  atomicMax(&totals[4], (unsigned long long)len);  // [4] = longest clique run
}

// K_pos.  One warp per query.  Similarities are computed from the SAME fp16 planes the tensor-core
// sweep consumes (hi*hi [+ hi*lo + lo*hi]) so thresholds and swept similarities agree to fp32
// accumulation noise; then rank-sorted ascending inside the warp (P_q is small: median 4, max ~360).
__global__ void __launch_bounds__(256) pos_thresholds_kernel(
    const __half* __restrict__ q_hi, const __half* __restrict__ q_lo, const __half* __restrict__ c_hi,
    const __half* __restrict__ c_lo, int d_pad, const int* __restrict__ q_i, int nq,
    const int* __restrict__ sorted_idx, const int* __restrict__ c_i, const int* __restrict__ seg_lo,
    const int* __restrict__ seg_len, const long long* __restrict__ off, float* __restrict__ raw,
    float* __restrict__ thr, float* __restrict__ lim, int* __restrict__ cnt) {
  const int q = (int)((blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5);
  const int lane = (int)(threadIdx.x & 31);
  if (q >= nq) return;
  const int first = seg_lo[q], len = seg_len[q], qi = q_i[q];
  const long long o = off[q];
  const uint4* qh = reinterpret_cast<const uint4*>(q_hi + (long long)q * d_pad);
  const uint4* ql = q_lo ? reinterpret_cast<const uint4*>(q_lo + (long long)q * d_pad) : nullptr;
  const int nvec = d_pad >> 3;  // 8 halves per 16-byte vector; d_pad is a multiple of 64
  int n = 0;
  for (int m = 0; m < len; ++m) {
    const int j = sorted_idx[first + m];
    if (c_i[j] == qi) continue;  // self / id collision
    const uint4* ch = reinterpret_cast<const uint4*>(c_hi + (long long)j * d_pad);
    const uint4* cl = c_lo ? reinterpret_cast<const uint4*>(c_lo + (long long)j * d_pad) : nullptr;
    float acc = 0.f;
    for (int v = lane; v < nvec; v += 32) {
      const uint4 a = qh[v], b = ch[v];
      const __half2* a2 = reinterpret_cast<const __half2*>(&a);
      const __half2* b2 = reinterpret_cast<const __half2*>(&b);
      uint4 al = make_uint4(0, 0, 0, 0), bl = make_uint4(0, 0, 0, 0);
      if (ql) { al = ql[v]; bl = cl[v]; }
      const __half2* al2 = reinterpret_cast<const __half2*>(&al);
      const __half2* bl2 = reinterpret_cast<const __half2*>(&bl);
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float2 fa = __half22float2(a2[e]), fb = __half22float2(b2[e]);
        acc = fmaf(fa.x, fb.x, acc);
        acc = fmaf(fa.y, fb.y, acc);
        if (ql) {
          const float2 fal = __half22float2(al2[e]), fbl = __half22float2(bl2[e]);
          acc = fmaf(fa.x, fbl.x, acc);
          acc = fmaf(fa.y, fbl.y, acc);
          acc = fmaf(fal.x, fb.x, acc);
          acc = fmaf(fal.y, fb.y, acc);
        }
      }
    }
    acc = warp_sum(acc);
    if (lane == 0) raw[o + n] = acc;
    ++n;
  }
  __syncwarp();
  // rank sort ascending: position = #{f : v_f < v_e or (v_f == v_e and f < e)}
  for (int e = lane; e < n; e += 32) {
    const float ve = raw[o + e];
    int r = 0;
    for (int f = 0; f < n; ++f) {
      const float vf = raw[o + f];
      r += (vf < ve) || (vf == ve && f < e);
    }
    thr[o + r] = ve;
  }
  __syncwarp();
  if (lane == 0) {
    cnt[q] = n;
    lim[q] = n > 0 ? thr[o] : __int_as_float(0x7f800000);
  }
}

// warp-level tensor-core tile D(16x8) += A(16x16, row major) * B(16x8, column major), fp16 in, fp32 accumulate
__device__ __forceinline__ void mma_16x8x16(float (&c)[4], const unsigned (&a)[4], const unsigned (&b)[2]) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}

// K_pos for chunked tracks (row f1).  One CTA (8 warps) per query track: for every relevant candidate track the kS x kS chunk
// similarities (same planes, same three products as the sweep) are reduced exactly like the sweep's epilogue does
// (red_inner over the candidate's chunks, red_outer over the query's), then rank-sorted ascending.
// The kS x kS blocks come from warp-level tensor-core tiles m16n8k16 read straight from the planes: the 16 tile ROWS
// are candidate chunks -- 16 / kS whole candidates per tile for kS <= 8 (eight two-chunk tracks, two eight-chunk
// tracks), one for kS = 16 -- and the 8 tile COLUMNS the query's chunks (two tiles for kS = 16), so a warp reads the
// query's rows once for all the candidates of its tile.  Two accumulators take alternate k windows (the dependent MMA
// chain is what bounds a warp).  Block b takes query track q_lo + b (a multi-GPU run gives every rank a share).
__global__ void __launch_bounds__(256) pos_thresholds_tracks_kernel(
    const __half* __restrict__ q_hi, const __half* __restrict__ q_lo, const __half* __restrict__ c_hi,
    const __half* __restrict__ c_lo, int d_pad, int ks, int red_inner, int red_outer, float red_scale,
    const int* __restrict__ q_i, int nq, const int* __restrict__ sorted_idx, const int* __restrict__ c_i,
    const int* __restrict__ seg_lo, const int* __restrict__ seg_len, const long long* __restrict__ off,
    float* __restrict__ raw, float* __restrict__ thr, float* __restrict__ lim, int* __restrict__ cnt,
    const int* __restrict__ q_len, const int* __restrict__ c_len, int q_first) {
  // its 8 warps take the relevant candidates tile by tile, round-robin (a clique of 160 versions is a handful of
  // sequential contractions per warp); slots of the query's CSR row are handed out by a shared counter
  const int q = q_first + (int)blockIdx.x;
  const int lane = (int)(threadIdx.x & 31), warp = (int)(threadIdx.x >> 5);
  __shared__ int n_sh;
  if (threadIdx.x == 0) n_sh = 0;
  __syncthreads();
  const int g = lane >> 2, tig = lane & 3;
  const int first = seg_lo[q], len = seg_len[q], qi = q_i[q];
  // ragged tracks (q_len / c_len given): valid chunks only, means over the valid counts -- same as the sweep's epilogue
  const bool ragged = c_len != nullptr;
  const int lq = ragged ? min(max(q_len[q], 1), ks) : ks;
  const long long o = off[q];
  const bool wide = ks > 8;                      // 16 chunks: one candidate fills the tile's rows, the query two tiles
  const int per = wide ? 1 : 16 / ks;            // candidates per tile
  const int kr = wide ? 8 : ks;                  // rows of one candidate inside an 8-row half of the tile
  // tile rows g and g + 8 of this lane: which candidate of the tile, which of its chunks
  const int sA = wide ? 0 : g / ks, cA = wide ? g : g % ks;
  const int sB = wide ? 0 : (g + 8) / ks, cB = wide ? g + 8 : (g + 8) % ks;
  const int ntile = wide ? 2 : 1;
  const float n_in = red_neutral(red_inner), n_out = red_neutral(red_outer);
  for (int m0 = warp * per; m0 < len; m0 += 8 * per) {
    const int mA = m0 + sA, mB = m0 + sB;
    const int jA = mA < len ? sorted_idx[first + mA] : -1;
    const int jB = mB < len ? sorted_idx[first + mB] : -1;
    const bool okA = jA >= 0 && c_i[jA] != qi, okB = jB >= 0 && c_i[jB] != qi;  // (self / id collision: not a candidate)
    const int lcA = (ragged && okA) ? min(max(c_len[jA], 1), ks) : ks;
    const int lcB = (ragged && okB) ? min(max(c_len[jB], 1), ks) : ks;
    const long long rA = ((long long)max(jA, 0) * ks + cA) * d_pad, rB = ((long long)max(jB, 0) * ks + cB) * d_pad;
    float wA = n_out, wB = n_out;   // outer reductions (over the query's chunks) of this lane's two rows' candidates
    for (int t = 0; t < ntile; ++t) {
      const long long rq = ((long long)q * ks + min(t * 8 + g, ks - 1)) * d_pad;  // B column g = query chunk t * 8 + g
      float c0[4] = {0.f, 0.f, 0.f, 0.f}, c1[4] = {0.f, 0.f, 0.f, 0.f};
      // (8 consecutive halves per lane, row and 32-wide k window: see pos_pairs_sorted_kernel; d_pad is a multiple of 64)
      for (int k = 0; k < d_pad; k += 64) {
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          float (&c)[4] = u ? c1 : c0;
          const int ko = k + u * 32 + tig * 8;
          const uint4 ah0 = __ldg(reinterpret_cast<const uint4*>(c_hi + rA + ko));
          const uint4 ah1 = __ldg(reinterpret_cast<const uint4*>(c_hi + rB + ko));
          const uint4 bh = __ldg(reinterpret_cast<const uint4*>(q_hi + rq + ko));
          const unsigned a1[4] = {ah0.x, ah1.x, ah0.y, ah1.y}, a2[4] = {ah0.z, ah1.z, ah0.w, ah1.w};
          const unsigned b1[2] = {bh.x, bh.y}, b2[2] = {bh.z, bh.w};
          mma_16x8x16(c, a1, b1);
          mma_16x8x16(c, a2, b2);
          if (q_lo) {
            const uint4 al0 = __ldg(reinterpret_cast<const uint4*>(c_lo + rA + ko));
            const uint4 al1 = __ldg(reinterpret_cast<const uint4*>(c_lo + rB + ko));
            const uint4 bl = __ldg(reinterpret_cast<const uint4*>(q_lo + rq + ko));
            const unsigned l1[4] = {al0.x, al1.x, al0.y, al1.y}, l2[4] = {al0.z, al1.z, al0.w, al1.w};
            const unsigned m1[2] = {bl.x, bl.y}, m2[2] = {bl.z, bl.w};
            mma_16x8x16(c, a1, m1);
            mma_16x8x16(c, a2, m2);
            mma_16x8x16(c, l1, b1);
            mma_16x8x16(c, l2, b2);
          }
        }
      }
      // c[0], c[1]: tile row g, query chunks t*8 + 2 tig, + 1;  c[2], c[3]: tile row g + 8, same columns
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        // inner: over the candidate's chunks = the rows of its slot (lanes that differ in the low bits of g; kS = 16: + the other half)
        float iA = cA < lcA ? c0[e] + c1[e] : n_in;
        float iB = cB < lcB ? c0[2 + e] + c1[2 + e] : n_in;
        if (wide) iA = red_op(iA, iB, red_inner);
        for (int x = 4; x < 4 * kr; x <<= 1) {
          iA = red_op(iA, __shfl_xor_sync(0xffffffffu, iA, x), red_inner);
          iB = red_op(iB, __shfl_xor_sync(0xffffffffu, iB, x), red_inner);
        }
        if (ragged) {
          if (red_inner == kRedSum) { iA *= 1.f / (float)lcA; iB *= 1.f / (float)lcB; }
        } else if (red_inner == kRedSum && red_outer != kRedSum) {
          iA *= red_scale;
          iB *= red_scale;
        }
        // outer: over the query's chunks = the tile's columns
        if (t * 8 + 2 * tig + e < lq) {
          wA = red_op(wA, iA, red_outer);
          wB = red_op(wB, iB, red_outer);
        }
      }
    }
#pragma unroll
    for (int x = 1; x < 4; x <<= 1) {
      wA = red_op(wA, __shfl_xor_sync(0xffffffffu, wA, x), red_outer);
      wB = red_op(wB, __shfl_xor_sync(0xffffffffu, wB, x), red_outer);
    }
    if (red_outer == kRedSum) {
      const float sc = ragged ? 1.f / (float)lq : red_scale;
      wA *= sc;
      wB *= sc;
    }
    // one writer per candidate: the lane of its first chunk's row (kS = 16: both halves belong to candidate A)
    if (tig == 0 && cA == 0 && okA) raw[o + atomicAdd(&n_sh, 1)] = wA;
    if (!wide && tig == 0 && cB == 0 && okB) raw[o + atomicAdd(&n_sh, 1)] = wB;
  }
  __syncthreads();
  const int n = n_sh;
  for (int e = (int)threadIdx.x; e < n; e += (int)blockDim.x) {
    const float ve = raw[o + e];
    int r = 0;
    for (int f = 0; f < n; ++f) {
      const float vf = raw[o + f];
      r += (vf < ve) || (vf == ve && f < e);
    }
    thr[o + r] = ve;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    cnt[q] = n;
    lim[q] = n > 0 ? thr[o] : __int_as_float(0x7f800000);
  }
}

// Multi-GPU staged K_pos of chunked tracks: after the ranks' threshold shares have been summed, every rank rebuilds the
// per-query values the sweep reads from the CSR offsets and the assembled thresholds, exactly as
// pos_thresholds_tracks_kernel writes them (a query's relevant candidates are the npos[q] = off[q + 1] - off[q]
// non-self members of its clique).  Integers never travel through the float all-reduce.
__global__ void track_limits_kernel(const long long* __restrict__ off, const float* __restrict__ thr, int nq,
                                    float* __restrict__ lim, int* __restrict__ cnt) {
  const int q = (int)(blockIdx.x * blockDim.x + threadIdx.x);
  if (q >= nq) return;
  const long long o = off[q];
  const int n = (int)(off[q + 1] - o);
  cnt[q] = n;
  lim[q] = n > 0 ? thr[o] : __int_as_float(0x7f800000);
}

// ---------------------------------------------------------------------------------------------------------
// Clique-sorted ("sorted space") view used by the symmetric all-vs-all sweep (eval_sym_epilogue.cuh)
// ---------------------------------------------------------------------------------------------------------
__global__ void gather_i32_kernel(const int* __restrict__ src, const int* __restrict__ idx, int n, int* __restrict__ dst) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) dst[t] = src[idx[t]];
}

// Tiles of the symmetric sweep that need id tests: row block rb x column tile t (t >= rb / 2) holds a self or
// same-clique pair iff the clique ranges of its rows and columns intersect (ids ascending in sorted space); ragged
// edge tiles are marked too (padded rows / columns must not be scored).
__global__ void dirty_clique_kernel(const int* __restrict__ s_c, int n, int n_row_blocks, int n_col_tiles,
                                    unsigned char* __restrict__ dirty) {
  const long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (idx >= (long long)n_row_blocks * n_col_tiles) return;
  const int rb = (int)(idx / n_col_tiles), t = (int)(idx - (long long)rb * n_col_tiles);
  if (t < (rb >> 1)) return;
  const int r0 = rb * kTileM, r1 = min(r0 + kTileM, n) - 1;
  const int c0 = t * kTileN, c1 = min(c0 + kTileN, n) - 1;
  const bool ragged = (r0 + kTileM > n) || (c0 + kTileN > n);
  const bool overlap = max(s_c[r0], s_c[c0]) <= min(s_c[r1], s_c[c1]);
  if (ragged || overlap) dirty[idx] = 1;
}

// Version-id collisions between different cliques can fall into any tile.  keys = version ids sorted ascending,
// pos = their sorted-space positions: every pair of equal keys marks the tile its (smaller, larger) position hits.
// A run longer than 16 equal ids (pathological input) marks everything.
__global__ void dirty_collision_kernel(const int* __restrict__ keys, const int* __restrict__ pos, int n,
                                       int n_row_blocks, int n_col_tiles, unsigned char* __restrict__ dirty,
                                       int* __restrict__ everything) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n || k == 0) return;
  const int key = keys[k];
  for (int b = 1; b <= 17 && k - b >= 0; ++b) {
    if (keys[k - b] != key) break;
    if (b == 17) { atomicExch(everything, 1); break; }
    const int p0 = min(pos[k], pos[k - b]), p1 = max(pos[k], pos[k - b]);
    dirty[(long long)(p0 / kTileM) * n_col_tiles + p1 / kTileN] = 1;
  }
  (void)n_row_blocks;
}

__global__ void dirty_everything_kernel(const int* __restrict__ everything, long long count, unsigned char* __restrict__ dirty) {
  const long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (idx < count && *everything) dirty[idx] = 1;
}

// K_pos in sorted space, step 1: similarities of every (query, relevant item) pair.  A clique is a contiguous run
// of rows, so the pairs of 16 consecutive queries form a dense 16 x |range| block of the Gram matrix around the
// diagonal: one CTA per 16-query block, each warp takes 8 candidates at a time and contracts the block with
// warp-level tensor-core MMAs (m16n8k16, fp32 accumulate) straight from the SAME fp16 planes the sweep consumes
// (hi*hi + hi*lo + lo*hi), 5-10x less L2 traffic than one dot product per pair.  Valid pairs (same clique, version
// ids differ) are appended to the query's CSR slice in arbitrary order (fill[q] counts them; step 2 sorts).

// kGather (all-vs-all through the rectangle sweep, e.g. with top-k): the planes are in the caller's row order, sorted
// row s is plane row perm[s], and off / fill are indexed by the caller's query index perm[q].
template <bool kGather>
__global__ void __launch_bounds__(256) pos_pairs_sorted_kernel(
    const __half* __restrict__ hi, const __half* __restrict__ lo, int d_pad, const int* __restrict__ s_c,
    const int* __restrict__ s_i, int n, const int* __restrict__ seg_lo, const int* __restrict__ seg_len,
    const long long* __restrict__ off, float* __restrict__ raw, int* __restrict__ fill,
    const int* __restrict__ perm = nullptr, int q_lo = 0, int q_hi = 0x7fffffff) {
  // [q_lo, q_hi): the queries this launch computes (multi-GPU: every rank takes a range of 16-query blocks, the
  // thresholds are then summed over the ranks -- the other ranks contribute zeros)
  auto plane_row = [&](int srow) { return kGather ? __ldg(perm + srow) : spread_plane_of(srow); };
  const int q0 = q_lo + blockIdx.x * 16;
  const int warp = (int)(threadIdx.x >> 5), lane = (int)(threadIdx.x & 31);
  const int g = lane >> 2, tig = lane & 3;
  const int qlast = min(q0 + 15, n - 1);
  const int lo_row = seg_lo[q0], hi_row = seg_lo[qlast] + seg_len[qlast];  // candidates any of the 16 queries needs
  const int qa = min(q0 + g, n - 1), qb = min(q0 + g + 8, n - 1);          // (clamped rows are discarded below)
  // (the planes are in the sweep's spread row order: sorted row s lives at plane row spread_plane_of(s))
  const int pa = plane_row(qa), pb = plane_row(qb);
  const __half* a_hi0 = hi + (long long)pa * d_pad;
  const __half* a_hi1 = hi + (long long)pb * d_pad;
  const __half* a_lo0 = lo ? lo + (long long)pa * d_pad : nullptr;
  const __half* a_lo1 = lo ? lo + (long long)pb * d_pad : nullptr;
  for (int j0 = lo_row + warp * 8; j0 < hi_row; j0 += 64) {
    const int jb = plane_row(min(j0 + g, n - 1));
    const __half* b_hi = hi + (long long)jb * d_pad;
    const __half* b_lo = lo ? lo + (long long)jb * d_pad : nullptr;
    float c[4] = {0.f, 0.f, 0.f, 0.f};
    // A dot product does not care in which order k is visited as long as A and B agree: every lane loads 8
    // CONSECUTIVE halves per row and 32-wide k window (one 16-byte access instead of four 4-byte ones) and feeds
    // them to two MMAs as if they were the fragment's (2 tig, 2 tig + 1, 2 tig + 8, 2 tig + 9) elements.
#pragma unroll 2
    for (int k = 0; k < d_pad; k += 32) {
      const int ko = k + tig * 8;
      const uint4 ah0 = __ldg(reinterpret_cast<const uint4*>(a_hi0 + ko)), ah1 = __ldg(reinterpret_cast<const uint4*>(a_hi1 + ko));
      const uint4 bh = __ldg(reinterpret_cast<const uint4*>(b_hi + ko));
      const unsigned a1[4] = {ah0.x, ah1.x, ah0.y, ah1.y}, a2[4] = {ah0.z, ah1.z, ah0.w, ah1.w};
      const unsigned b1[2] = {bh.x, bh.y}, b2[2] = {bh.z, bh.w};
      mma_16x8x16(c, a1, b1);
      mma_16x8x16(c, a2, b2);
      if (lo) {
        const uint4 al0 = __ldg(reinterpret_cast<const uint4*>(a_lo0 + ko)), al1 = __ldg(reinterpret_cast<const uint4*>(a_lo1 + ko));
        const uint4 bl = __ldg(reinterpret_cast<const uint4*>(b_lo + ko));
        const unsigned l1[4] = {al0.x, al1.x, al0.y, al1.y}, l2[4] = {al0.z, al1.z, al0.w, al1.w};
        const unsigned m1[2] = {bl.x, bl.y}, m2[2] = {bl.z, bl.w};
        mma_16x8x16(c, a1, m1);
        mma_16x8x16(c, a2, m2);
        mma_16x8x16(c, l1, b1);
        mma_16x8x16(c, l2, b2);
      }
    }
    // c[0], c[1]: query q0 + g, candidates j0 + 2 tig, + 1;  c[2], c[3]: query q0 + g + 8, same candidates
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int q = q0 + g + (e >> 1) * 8;
      const int j = j0 + tig * 2 + (e & 1);
      if (q < n && q < q_hi && j < hi_row && s_c[q] == s_c[j] && s_i[q] != s_i[j]) {
        const int oq = kGather ? __ldg(perm + q) : q;
        const int slot = atomicAdd(fill + oq, 1);
        raw[off[oq] + slot] = c[e];
      }
    }
  }
}

// K_pos step 2 for the rectangle sweep after pos_pairs_sorted_kernel<true>: one warp per query rank-sorts the cnt[q]
// appended similarities ascending into thr and sets lim[q] (the lowest, +inf if none).
__global__ void __launch_bounds__(256) pos_sort_kernel(int nq, const long long* __restrict__ off, const float* __restrict__ raw,
                                                       float* __restrict__ thr, float* __restrict__ lim,
                                                       const int* __restrict__ cnt) {
  const int q = (int)((blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5);
  const int lane = (int)(threadIdx.x & 31);
  if (q >= nq) return;
  const int n = cnt[q];
  const long long o = off[q];
  for (int e = lane; e < n; e += 32) {
    const float ve = raw[o + e];
    int r = 0;
    for (int f = 0; f < n; ++f) {
      const float vf = raw[o + f];
      r += (vf < ve) || (vf == ve && f < e);
    }
    thr[o + r] = ve;
  }
  __syncwarp();
  if (lane == 0) lim[q] = n > 0 ? thr[o] : __int_as_float(0x7f800000);
}

// K_pos step 2.  One warp per query: rank-sort its pair similarities ascending into thr (CSR); the lowest four go
// to lvl[q] (+inf padded), {offset, count} to cinfo[q].  Rows q >= n (padding up to a whole column tile) get
// lvl = +inf, cinfo = {total, 0}.
__global__ void __launch_bounds__(256) pos_sort_sorted_kernel(const int* __restrict__ npos, int n, int n_padded,
                                                              const long long* __restrict__ off,
                                                              const float* __restrict__ raw, float* __restrict__ thr,
                                                              int* __restrict__ cnt, float4* __restrict__ lvl,
                                                              uint2* __restrict__ cinfo, int q_lo = 0, int q_hi = 0x7fffffff,
                                                              int partial = 0) {
  // partial (wealy_eval_run_host: the queries arrive range by range): the grid covers [q_lo, n_padded) and touches
  // nothing outside [q_lo, q_hi) -- the other ranges are written by their own launches; the padding rows belong to the
  // range that reaches n
  const int q = (partial ? q_lo : 0) + (int)((blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5);
  const int lane = (int)(threadIdx.x & 31);
  if (q >= n_padded) return;
  if (partial && (q < n ? q >= q_hi : q_hi < n)) return;
  const float inf = __int_as_float(0x7f800000);
  const int pq = spread_plane_of(q);  // lvl / cinfo are read by plane row (per-tile bulk copies of the sweep)
  if (q < n && (q < q_lo || q >= q_hi)) {
    // another rank's query: id-only data here, zeros where the sum over the ranks will put that rank's thresholds
    if (lane == 0) {
      cnt[q] = npos[q];
      lvl[pq] = make_float4(0.f, 0.f, 0.f, 0.f);
      cinfo[pq] = make_uint2((unsigned)off[q], (unsigned)npos[q]);
    }
    return;
  }
  if (q >= n) {
    if (lane == 0) {
      lvl[pq] = make_float4(inf, inf, inf, inf);
      cinfo[pq] = make_uint2((unsigned)off[n], 0u);
    }
    return;
  }
  const int np = npos[q];
  const long long o = off[q];
  // rank sort ascending: position = #{f : v_f < v_e or (v_f == v_e and f < e)}
  for (int e = lane; e < np; e += 32) {
    const float ve = raw[o + e];
    int r = 0;
    for (int f = 0; f < np; ++f) {
      const float vf = raw[o + f];
      r += (vf < ve) || (vf == ve && f < e);
    }
    thr[o + r] = ve;
  }
  __syncwarp();
  if (lane == 0) {
    cnt[q] = np;
    lvl[pq] = make_float4(np > 0 ? thr[o] : inf, np > 1 ? thr[o + 1] : inf, np > 2 ? thr[o + 2] : inf,
                          np > 3 ? thr[o + 3] : inf);
    cinfo[pq] = make_uint2((unsigned)o, (unsigned)np);
  }
}

// K2.  One warp per query; warp-shuffle suffix scan over the rank histogram.
//   above[r]    = sum_{m >= r} hist[m]            negatives ranked above the r-th lowest relevant item
//   rank_all[r] = 1 + above[r] + (P - 1 - r)      relevant items above it are the ones sorted after it
//   rank_rel[r] = P - r
//   AP = 1/P sum_r rank_rel[r] / rank_all[r],  R1 = rank_all[P-1]
__global__ void __launch_bounds__(256) ap_reduce_kernel(const unsigned int* __restrict__ hist,
                                                        const long long* __restrict__ off,
                                                        const int* __restrict__ cnt, int nq, float* __restrict__ ap,
                                                        float* __restrict__ r1, double* __restrict__ sums,
                                                        const int* __restrict__ perm = nullptr) {
  const int q = (int)((blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5);
  const int lane = (int)(threadIdx.x & 31);
  const bool live = q < nq;  // (no early return: the block reduces the running sums together)
  const int P = live ? cnt[q] : 0;
  const unsigned int* h = hist + (live ? off[q] : 0);
  float acc = 0.f;
  unsigned int carry = 0;  // negatives above everything processed so far (higher r)
  float first_rank = 0.f;
  for (int base = P - 1; base >= 0; base -= 32) {
    const int r = base - lane;  // lane 0 takes the highest remaining r
    unsigned int v = r >= 0 ? h[r] : 0u;
    // inclusive scan over lanes (lane l gets sum of lanes 0..l) == suffix sum over r
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned int t = __shfl_up_sync(0xffffffffu, v, o);
      if (lane >= o) v += t;
    }
    const unsigned int above = carry + v;
    if (r >= 0) {
      const float rank_all = 1.f + (float)above + (float)(P - 1 - r);
      acc += (float)(P - r) / rank_all;
      if (r == P - 1) first_rank = rank_all;
    }
    carry += __shfl_sync(0xffffffffu, v, 31);
  }
  acc = warp_sum(acc);
  first_rank = warp_max(first_rank);
  double s_ap = 0.0, s_r1 = 0.0, s_n = 0.0;
  if (lane == 0 && live) {
    const float a = P > 0 ? acc / (float)P : __int_as_float(0x7fc00000);
    const float f = P > 0 ? first_rank : __int_as_float(0x7fc00000);
    const int dst = perm ? perm[q] : q;  // sorted space -> the caller's row order
    ap[dst] = a;
    r1[dst] = f;
    if (P > 0) {
      s_ap = (double)a;
      s_r1 = (double)f;
      s_n = 1.0;
    }
  }
  // running sums for MAP / MR1: one atomic triple per block, not per query (same-address atomics serialise)
  __shared__ double part[3][8];
  const int w = (int)(threadIdx.x >> 5);
  if (lane == 0) {
    part[0][w] = s_ap;
    part[1][w] = s_r1;
    part[2][w] = s_n;
  }
  __syncthreads();
  if (threadIdx.x < 3) {
    double t = 0.0;
    for (int k = 0; k < 8; ++k) t += part[threadIdx.x][k];
    if (t != 0.0) atomicAdd(&sums[threadIdx.x], t);
  }
}

// Per-item ranks (what AP is made of), exported for callers / parity tests: for every query, its relevant items
// best first -- rank_all (1-based rank among all non-self candidates) and similarity.  Same suffix scan as K2.
// `off` / `cnt` are in the order of the last sweep (sorted space when perm != nullptr), `out_off` is the CSR of
// the caller's query order.
__global__ void __launch_bounds__(256) rank_export_kernel(const unsigned int* __restrict__ hist, const float* __restrict__ thr,
                                                          const long long* __restrict__ off, const int* __restrict__ cnt,
                                                          int nq, const long long* __restrict__ out_off,
                                                          const int* __restrict__ perm, int* __restrict__ ranks,
                                                          float* __restrict__ sims) {
  const int q = (int)((blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5);
  const int lane = (int)(threadIdx.x & 31);
  if (q >= nq) return;
  const int P = cnt[q];
  const long long o = off[q];
  const long long oo = out_off[perm ? perm[q] : q];
  unsigned int carry = 0;
  for (int base = P - 1; base >= 0; base -= 32) {
    const int r = base - lane;
    unsigned int v = r >= 0 ? hist[o + r] : 0u;
#pragma unroll
    for (int s = 1; s < 32; s <<= 1) {
      const unsigned int t = __shfl_up_sync(0xffffffffu, v, s);
      if (lane >= s) v += t;
    }
    if (r >= 0) {
      ranks[oo + (P - 1 - r)] = (int)(1u + carry + v + (unsigned)(P - 1 - r));
      sims[oo + (P - 1 - r)] = thr[o + r];
    }
    carry += __shfl_sync(0xffffffffu, v, 31);
  }
}

// K3.  One warp per query: gather the candidates of every part, keep the k best (descending
// similarity, ties -> lower candidate index, like a stable ascending-distance argsort).
__global__ void __launch_bounds__(256) topk_finalize_kernel(const float* __restrict__ cand_val,
                                                            const int* __restrict__ cand_idx,
                                                            const int* __restrict__ cand_cnt, int parts, int nq,
                                                            int cap, int k, long long* __restrict__ out_idx,
                                                            float* __restrict__ out_sim) {
  const int q = (int)((blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5);
  const int lane = (int)(threadIdx.x & 31);
  if (q >= nq) return;
  for (int e = lane; e < k; e += 32) {
    out_idx[(long long)q * k + e] = -1;
    out_sim[(long long)q * k + e] = __int_as_float(0xff800000);
  }
  __syncwarp();
  for (int p = 0; p < parts; ++p) {
    const long long b = ((long long)p * nq + q) * cap;
    const int n = cand_cnt[(long long)p * nq + q];
    for (int e = lane; e < n; e += 32) {
      const float ve = cand_val[b + e];
      const int ie = cand_idx[b + e];
      int r = 0;
      for (int p2 = 0; p2 < parts && r < k; ++p2) {
        const long long b2 = ((long long)p2 * nq + q) * cap;
        const int n2 = cand_cnt[(long long)p2 * nq + q];
        for (int f = 0; f < n2; ++f) {
          const float vf = cand_val[b2 + f];
          r += (vf > ve) || (vf == ve && cand_idx[b2 + f] < ie);
        }
      }
      if (r < k) {
        out_idx[(long long)q * k + r] = ie;
        out_sim[(long long)q * k + r] = ve;
      }
    }
  }
}


// K3 (fast path: the <= 4 candidate lists of a query hold <= 1536 entries in total, i.e. k <= ~190): one warp per query gathers every part's
// candidates into registers, selects the k best in O(n) (warp_select_topk), then orders the k
// survivors by rank counting (k^2 / 32 steps) -- descending similarity, ties -> lower index.
constexpr int kFinPerLane = 48;  // up to 1536 gathered candidates (4 lists of 384)
__global__ void __launch_bounds__(128) topk_finalize_select_kernel(const float* __restrict__ cand_val,
                                                                   const int* __restrict__ cand_idx,
                                                                   const int* __restrict__ cand_cnt, int parts, int nq,
                                                                   int cap, int k, float* __restrict__ stage_val,
                                                                   int* __restrict__ stage_idx,
                                                                   long long* __restrict__ out_idx,
                                                                   float* __restrict__ out_sim) {
  const int q = (int)((blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5);
  const int lane = (int)(threadIdx.x & 31);
  if (q >= nq) return;
  // staging area of this query: [parts * cap] contiguous (value, index) pairs
  float* sv = stage_val + (long long)q * parts * cap;
  int* si = stage_idx + (long long)q * parts * cap;
  int n = 0;
  for (int p = 0; p < parts; ++p) {
    const long long b = ((long long)p * nq + q) * cap;
    const int np = cand_cnt[(long long)p * nq + q];
    for (int e = lane; e < np; e += 32) {
      sv[n + e] = cand_val[b + e];
      si[n + e] = cand_idx[b + e];
    }
    n += np;
  }
  const int kk = min(k, n);
  if (n > kk) warp_select_topk<kFinPerLane>(sv, si, n, kk, lane);
  __syncwarp();
  for (int e = lane; e < k; e += 32) {
    if (e >= kk) {
      out_idx[(long long)q * k + e] = -1;
      out_sim[(long long)q * k + e] = __int_as_float(0xff800000);
    }
  }
  for (int e = lane; e < kk; e += 32) {
    const float ve = sv[e];
    const int ie = si[e];
    int r = 0;
    for (int f = 0; f < kk; ++f) {
      const float vf = sv[f];
      r += (vf > ve) || (vf == ve && si[f] < ie);
    }
    out_idx[(long long)q * k + r] = ie;
    out_sim[(long long)q * k + r] = ve;
  }
}

}  // namespace wealy
