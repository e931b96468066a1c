// Warp-specialised sm_100a contraction core shared by every hot kernel of the path.
//
//   S[r, c] = sum_k A[r, k] * B[c, k]        A = query rows, B = candidate rows, both K-major fp16
//
// * operands are the fp16 "planes" written by the prep kernel: a `hi` plane and (3-pass parity
//   mode) a `lo` residual plane; one pipeline stage holds {A_hi, A_lo, B_hi, B_lo} for one
//   k-block and feeds three tcgen05.mma groups: hi*hi + hi*lo + lo*hi (fp32-grade accuracy from
//   fp16 tensor cores, loading 4 tiles instead of the 6 a K'=3D GEMM would);
// * TMA (128B/64B swizzle) -> shared-memory ring -> tcgen05.mma (M=128, N=256, K=16) issued by
//   one thread -> two 256-column TMEM accumulators so the epilogue of tile t overlaps the MMAs
//   of tile t+1;
// * the N x N matrix is never written by this core: the accumulator is handed to an Epilogue
//   policy 32 columns at a time, one accumulator row (= one query) per thread.
//
// Work decomposition: a *unit* is (row block of 128 queries) x (chunk of consecutive column
// tiles).  Units are dealt round-robin to a persistent grid so that concurrently resident CTAs
// sweep the same column chunk (candidate tiles are then shared through the 126 MB L2).
#pragma once
#include "ptx.cuh"

namespace wealy {

constexpr int kTileM = 128;   // queries per tile (TMEM lanes)
constexpr int kTileN = 256;   // candidates per tile (TMEM columns per accumulator)
constexpr int kUmmaK = 16;    // K per tcgen05.mma for 16-bit inputs
constexpr int kChunkCols = 32;  // columns handed to the epilogue per tcgen05.ld

// "Spread" row order of the symmetric evaluation sweep.  In clique-sorted order equally hot rows are neighbours, and a
// TMEM lane quadrant (32 consecutive accumulator rows = one pair of epilogue warps) would own a run of them and gate
// the whole CTA.  The operand planes (and every per-row array the sweep reads) are therefore stored with the rows of
// each 128-row block dealt round-robin to the four quadrants: plane row p of a block holds sorted row
// 4 * (p % 32) + p / 32 of that block.  Blocks are unchanged as sets, so tiles, clique ranges and CSR slices are too.
__host__ __device__ __forceinline__ int spread_sorted_of(int p) {
  const int r = p & 127;
  return (p & ~127) + ((r & 31) << 2) + (r >> 5);
}
__host__ __device__ __forceinline__ int spread_plane_of(int s) {
  const int u = s & 127;
  return (s & ~127) + ((u & 3) << 5) + (u >> 2);
}

struct GemmTmaps {
  CUtensorMap a_hi, a_lo, b_hi, b_lo;
};

struct GemmShape {
  int m_rows;           // valid query rows
  int n_cols;           // valid candidate columns
  int k_blocks;         // number of kBlockK-wide k-blocks (planes are zero padded)
  int n_row_blocks;     // ceil(m_rows / 128)
  int n_col_tiles;      // ceil(n_cols / 256)
  int tiles_per_chunk;  // column tiles per unit
  int n_col_chunks;     // ceil(n_col_tiles / tiles_per_chunk)
  int group_rows;       // row blocks per scheduling group (see decode_unit)
  int* unit_counter;    // global work counter of this launch: dynamic unit scheduling.  unit_counter[1] counts the
                        //   CTAs that are through; the last one zeroes both again, so the host never has to (no memset
                        //   in front of every launch; the slots start out zero)
  int sym;              // CTA-pair core (gemm_core2.cuh) only -- bit 0: symmetric all-vs-all, only tiles that reach
                        //   above the diagonal are computed; bit 1: the pair's CTAs take alternate rows
  int rb_stride;        // multi-GPU symmetric sweep: this launch owns row blocks rb_offset + k * rb_stride
  int rb_offset;        //   (n_row_blocks counts the owned ones)
  // column-tile window of this launch: only tiles in [win0, win1) and outside [skip0, skip1) are contracted (the
  // data-parallel losses sweep the rank's own column block while the other ranks' rows are still in flight, then
  // everything but that block); the defaults of fill_shape select every tile
  int win0, win1, skip0, skip1;
};

__device__ __forceinline__ bool tile_selected(const GemmShape& sh, int t) {
  return t >= sh.win0 && t < sh.win1 && !(t >= sh.skip0 && t < sh.skip1);
}

// Unit order.  Units are handed out in sequence from a global atomic counter (the TMA warp fetches the
// next index and publishes it to the MMA and epilogue warps through a 2-deep shared-memory mailbox), so
// ~148 consecutive units run together and CTAs cannot drift apart by more than one unit -- which is
// what keeps the candidate tiles they share alive in L2.  Units are enumerated group by group: a group is `group_rows` row blocks x ALL column
// chunks, chunk-major inside the group.  With group_rows = #SMs / #chunks the CTAs resident together
// cover few row blocks (their query tiles, re-read once per column tile, are the L2 working set:
// 37 x 512 KB instead of 148 x 512 KB at C2) while each chunk's candidate tiles are still shared by
// group_rows CTAs sweeping it in step.
__device__ __forceinline__ void decode_unit(const GemmShape& sh, int u, int& chunk, int& rb) {
  const int per_group = sh.group_rows * sh.n_col_chunks;
  const int g = u / per_group;
  const int within = u - g * per_group;
  const int rows_here = min(sh.group_rows, sh.n_row_blocks - g * sh.group_rows);
  chunk = within / rows_here;
  rb = (g * sh.group_rows + (within - chunk * rows_here)) * sh.rb_stride + sh.rb_offset;
}

// Every CTA calls this once, after its last fetch from the unit counter: the last CTA through resets the pair of
// counters for the slot's next launch (stream order makes the reset visible to it).
__device__ __forceinline__ void release_unit_counter(const GemmShape& sh) {
  if (threadIdx.x == 0) {
    const int done = atomicAdd(sh.unit_counter + 1, 1);
    if (done == (int)gridDim.x - 1) {
      sh.unit_counter[0] = 0;
      sh.unit_counter[1] = 0;
    }
  }
}

template <int kPasses, int kBlockK>
struct GemmSmem {
  static constexpr int kSwizzle = kBlockK * 2;  // bytes per smem row == swizzle span
  static constexpr int kABytes = kTileM * kBlockK * 2;
  static constexpr int kBBytes = kTileN * kBlockK * 2;
  static constexpr int kPlanes = kPasses == 3 ? 2 : 1;
  static constexpr int kStageBytes = kPlanes * (kABytes + kBBytes);
  static constexpr int kBudget = 227 * 1024 - 2048 - 30 * 1024;  // alignment slack + barriers + epilogue scratch
  static constexpr int kMaxStages = 8;
  static constexpr int kStages = (kBudget / kStageBytes) > kMaxStages ? kMaxStages : (kBudget / kStageBytes);
  static constexpr int kBarBytes = 512;
  static constexpr int kCore = kStages * kStageBytes + kBarBytes;  // + per-warp epilogue scratch + 1024 align slack
  static_assert(kStages >= 2, "need at least a double-buffered ring");
  static constexpr int total(int epi_warps, int scratch_per_warp, int cta_scratch) {
    return kCore + epi_warps * scratch_per_warp + cta_scratch + 1024;
  }
};

// What the core hands to an epilogue policy besides the accumulator.
struct EpiCtx {
  uint8_t* warp_scratch;  // Epi::kWarpScratchBytes of shared memory private to this epilogue warp
  uint8_t* cta_scratch;   // Epi::kCtaScratchBytes shared by all epilogue warps of the CTA
  int tid;                // thread index inside the epilogue group, [0, nthreads)
  int nthreads;           // epilogue threads per CTA (named barrier 1 is reserved for them)
  int row_base;           // first query row of the unit's row block (of the 256-row super block in the CTA-pair core)
  int row_span;           // consecutive rows [row_base, row_base + row_span) this CTA's rows are drawn from (128, or 256)
  int first_col;          // first column this warp will see in the unit ...
  int col_step;           // ... and the distance to the column of its next chunk
  const uint8_t* col_slot;  // Epi::kColSlots > 0: this tile's per-column data (bulk-copied by the TMA thread)
};

// Epilogues that want per-tile column data staged in shared memory declare kColSlots / kColSlotBytes /
// kOffColSlots (offset inside their CTA scratch) and col_bulk_src(); the others get these defaults.
template <class Epi, class = void>
struct ColSlotTraits {
  static constexpr int kSlots = 0, kBytes = 0, kOffset = 0;
};
template <class Epi>
struct ColSlotTraits<Epi, decltype((void)Epi::kColSlots)> {
  static constexpr int kSlots = Epi::kColSlots, kBytes = Epi::kColSlotBytes, kOffset = Epi::kOffColSlots;
};

// Epilogue policy contract (all __device__, called by the epilogue warps only; every epilogue
// thread calls row_begin / row_end exactly once per unit, so they may use the group barrier):
//   struct Params;                      POD passed by value to the kernel
//   struct RowState;                    per-thread state that lives across one unit
//   static constexpr int kWarpScratchBytes, kCtaScratchBytes;   shared-memory scratch (may be 0)
//   static void row_begin(const Params&, RowState&, int row, int part, const GemmShape&, const EpiCtx&);
//   static void chunk32(const Params&, RowState&, int row, int col0, const uint32_t (&acc)[32], const GemmShape&,
//                       const EpiCtx&);
//   static void tile_begin(const Params&, RowState&, const GemmShape&, const EpiCtx&, int tile);  before the accumulator wait
//   static void tile_end(const Params&, RowState&, const GemmShape&, const EpiCtx&);   after the accumulator is released
//   static void row_end(const Params&, RowState&, int row, int part, const GemmShape&, const EpiCtx&);
// `row` is the global query row owned by the thread, `part` identifies the partial result slot
// (column chunk x epilogue half) when a row is split over several units / warps.

template <class Epi, int kPasses, int kBlockK, int kEpiWarps>
__global__ void __launch_bounds__(64 + kEpiWarps * 32, 1)
gemm_kernel(const __grid_constant__ GemmTmaps tmaps, const GemmShape shape, const typename Epi::Params ep) {
  using SM = GemmSmem<kPasses, kBlockK>;
  constexpr int kStages = SM::kStages;
  constexpr int kHalves = kEpiWarps / 4;  // epilogue warps per TMEM lane quadrant
  static_assert(kEpiWarps == 4 || kEpiWarps == 8 || kEpiWarps == 12 || kEpiWarps == 16, "4, 8, 12 or 16 epilogue warps");
  static_assert(kPasses == 1 || kPasses == 3, "1 (fp16) or 3 (fp16 hi/lo) passes");

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* bar_base = smem + kStages * SM::kStageBytes;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(bar_base);
  uint64_t* empty_bar = full_bar + kStages;
  uint64_t* tmem_full = empty_bar + kStages;
  uint64_t* tmem_empty = tmem_full + 2;
  uint64_t* unit_full = tmem_empty + 2;
  uint64_t* unit_empty = unit_full + 2;
  using CS = ColSlotTraits<Epi>;
  constexpr int kColSlots = CS::kSlots;
  uint64_t* col_full = unit_empty + 2;
  uint64_t* col_empty = col_full + (kColSlots > 0 ? kColSlots : 1);
  int* unit_slot = reinterpret_cast<int*>(col_empty + (kColSlots > 0 ? kColSlots : 1));
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(unit_slot + 2);
  static_assert((2 * kStages + 8 + 2 * (kColSlots > 0 ? kColSlots : 1)) * 8 + 16 <= SM::kBarBytes, "barrier area");
  uint8_t* scratch_base = bar_base + SM::kBarBytes;
  uint8_t* col_slots = scratch_base + kEpiWarps * Epi::kWarpScratchBytes + CS::kOffset;

  const int warp_idx = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const int lane = (int)ptx::lane_id();

  if (warp_idx == 0 && lane == 0) {
    ptx::prefetch_tensormap(&tmaps.a_hi);
    ptx::prefetch_tensormap(&tmaps.b_hi);
    if (kPasses == 3) {
      ptx::prefetch_tensormap(&tmaps.a_lo);
      ptx::prefetch_tensormap(&tmaps.b_lo);
    }
    for (int s = 0; s < kStages; ++s) {
      ptx::mbar_init(&full_bar[s], 1);
      ptx::mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      ptx::mbar_init(&tmem_full[a], 1);
      ptx::mbar_init(&tmem_empty[a], kEpiWarps);
      ptx::mbar_init(&unit_full[a], 1);
      ptx::mbar_init(&unit_empty[a], 1 + kEpiWarps);  // MMA thread + one lane per epilogue warp
    }
    for (int c = 0; c < kColSlots; ++c) {
      ptx::mbar_init(&col_full[c], 1);
      ptx::mbar_init(&col_empty[c], kEpiWarps);
    }
    ptx::fence_mbar_init();
  }
  if (warp_idx == 1) ptx::tmem_alloc<512>(tmem_slot);
  ptx::tc_fence_before_sync();
  __syncthreads();
  ptx::tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;

  const int n_units = shape.n_row_blocks * shape.n_col_chunks;

  if (warp_idx == 0) {
    // ===================================================== TMA producer (one thread)
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      int us = 0;
      uint32_t uphase = 0;
      int cs = 0;
      uint32_t cphase = 0;
      while (true) {
        // fetch the next unit and publish it to the MMA / epilogue warps
        ptx::mbar_wait(&unit_empty[us], uphase ^ 1u);
        int u = atomicAdd(shape.unit_counter, 1);
        if (u >= n_units) u = -1;
        unit_slot[us] = u;
        ptx::mbar_arrive(&unit_full[us]);
        if (++us == 2) { us = 0; uphase ^= 1u; }
        if (u < 0) break;
        int chunk, rb;
        decode_unit(shape, u, chunk, rb);
        const int t1 = min((chunk + 1) * shape.tiles_per_chunk, shape.n_col_tiles);
        const int t0 = chunk * shape.tiles_per_chunk;
        for (int t = t0; t < t1; ++t) {
          if (!tile_selected(shape, t)) continue;
          if constexpr (kColSlots > 0) {
            // per-tile column data of the epilogue: contiguous arrays indexed by column -> 1-D bulk copies
            ptx::mbar_wait(&col_empty[cs], cphase ^ 1u);
            const void *s0, *s1;
            Epi::col_bulk_src(ep, t, s0, s1);
            uint8_t* dst = col_slots + cs * CS::kBytes;
            ptx::mbar_expect_tx(&col_full[cs], CS::kBytes);
            ptx::bulk_load(dst, s0, Epi::kLvlBytes, &col_full[cs]);
            ptx::bulk_load(dst + Epi::kLvlBytes, s1, CS::kBytes - Epi::kLvlBytes, &col_full[cs]);
            if (++cs == kColSlots) { cs = 0; cphase ^= 1u; }
          }
          for (int kb = 0; kb < shape.k_blocks; ++kb) {
            ptx::mbar_wait(&empty_bar[stage], phase ^ 1u);
            uint8_t* st = smem + stage * SM::kStageBytes;
            ptx::mbar_expect_tx(&full_bar[stage], SM::kStageBytes);
            // the CTA's query tiles are re-read once per column tile of the unit (~100x): the 148
            // resident row blocks (76 MB in fp16x3) are the L2 working set -> evict_last; a candidate
            // tile only has to survive until every CTA of the wave has passed it -> normal priority
            ptx::tma_load_2d(st, &tmaps.a_hi, &full_bar[stage], kb * kBlockK, rb * kTileM, ptx::kEvictLast);
            ptx::tma_load_2d(st + SM::kPlanes * SM::kABytes, &tmaps.b_hi, &full_bar[stage], kb * kBlockK,
                             t * kTileN, ptx::kEvictNormal);
            if (kPasses == 3) {
              ptx::tma_load_2d(st + SM::kABytes, &tmaps.a_lo, &full_bar[stage], kb * kBlockK, rb * kTileM,
                               ptx::kEvictLast);
              ptx::tma_load_2d(st + 2 * SM::kABytes + SM::kBBytes, &tmaps.b_lo, &full_bar[stage], kb * kBlockK,
                               t * kTileN, ptx::kEvictNormal);
            }
            if (++stage == kStages) { stage = 0; phase ^= 1u; }
          }
        }
      }
    }
  } else if (warp_idx == 1) {
    // ===================================================== MMA issuer (one thread)
    if (lane == 0) {
      constexpr uint32_t idesc = ptx::make_idesc_f16(kTileM, kTileN, false);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      int us = 0;
      uint32_t uphase = 0;
      while (true) {
        ptx::mbar_wait(&unit_full[us], uphase);
        const int u = unit_slot[us];
        ptx::mbar_arrive(&unit_empty[us]);
        if (++us == 2) { us = 0; uphase ^= 1u; }
        if (u < 0) break;
        int chunk, rb;
        decode_unit(shape, u, chunk, rb);
        const int t1 = min((chunk + 1) * shape.tiles_per_chunk, shape.n_col_tiles);
        const int t0 = chunk * shape.tiles_per_chunk;
        for (int t = t0; t < t1; ++t) {
          if (!tile_selected(shape, t)) continue;
          ptx::mbar_wait(&tmem_empty[acc], acc_phase ^ 1u);  // epilogue has drained this accumulator
          ptx::tc_fence_after_sync();
          const uint32_t d_tmem = tmem_base + (uint32_t)(acc * kTileN);
          for (int kb = 0; kb < shape.k_blocks; ++kb) {
            ptx::mbar_wait(&full_bar[stage], phase);
            ptx::tc_fence_after_sync();
            const uint32_t st = ptx::smem_u32(smem + stage * SM::kStageBytes);
            const uint64_t a_hi = ptx::make_smem_desc<SM::kSwizzle>(st);
            const uint64_t b_hi = ptx::make_smem_desc<SM::kSwizzle>(st + SM::kPlanes * SM::kABytes);
            const uint64_t a_lo = ptx::make_smem_desc<SM::kSwizzle>(st + SM::kABytes);
            const uint64_t b_lo = ptx::make_smem_desc<SM::kSwizzle>(st + 2 * SM::kABytes + SM::kBBytes);
#pragma unroll
            for (int kk = 0; kk < kBlockK / kUmmaK; ++kk) {
              const uint64_t adv = (uint64_t)((kk * kUmmaK * 2) >> 4);  // +32 B inside the swizzle span
              ptx::umma_f16(d_tmem, a_hi + adv, b_hi + adv, idesc, (uint32_t)((kb | kk) != 0));
              if (kPasses == 3) {
                ptx::umma_f16(d_tmem, a_hi + adv, b_lo + adv, idesc, 1u);
                ptx::umma_f16(d_tmem, a_lo + adv, b_hi + adv, idesc, 1u);
              }
            }
            ptx::umma_commit(&empty_bar[stage]);  // smem slot reusable once these MMAs retire
            if (kb == shape.k_blocks - 1) ptx::umma_commit(&tmem_full[acc]);
            if (++stage == kStages) { stage = 0; phase ^= 1u; }
          }
          if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
        }
      }
    }
  } else {
    // ===================================================== epilogue warps
    const int ew = warp_idx - 2;
    const int quad = warp_idx & 3;          // TMEM lane quadrant this warp may read
    const int half = kHalves == 1 ? 0 : (ew >> 2);
    const int row_in_tile = quad * 32 + lane;
    int acc = 0;
    uint32_t acc_phase = 0;
    int us = 0;
    uint32_t uphase = 0;
    int cs = 0;
    uint32_t cphase = 0;
    while (true) {
      ptx::mbar_wait_warp(&unit_full[us], uphase);
      const int u = unit_slot[us];
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&unit_empty[us]);
      if (++us == 2) { us = 0; uphase ^= 1u; }
      if (u < 0) break;
      int chunk, rb;
      decode_unit(shape, u, chunk, rb);
      const int t1 = min((chunk + 1) * shape.tiles_per_chunk, shape.n_col_tiles);
      const int t0 = chunk * shape.tiles_per_chunk;
      const int row = rb * kTileM + row_in_tile;
      const int part = chunk * kHalves + half;
      typename Epi::RowState rs;
      EpiCtx ctx;
      ctx.warp_scratch = scratch_base + ew * Epi::kWarpScratchBytes;
      ctx.cta_scratch = scratch_base + kEpiWarps * Epi::kWarpScratchBytes;
      ctx.tid = ew * 32 + lane;
      ctx.nthreads = kEpiWarps * 32;
      ctx.row_base = rb * kTileM;
      ctx.row_span = kTileM;
      ctx.first_col = t0 * kTileN + half * kChunkCols;
      ctx.col_step = kHalves * kChunkCols;
      ctx.col_slot = nullptr;
      Epi::row_begin(ep, rs, row, part, shape, ctx);
      for (int t = t0; t < t1; ++t) {
        if (!tile_selected(shape, t)) continue;
        if constexpr (kColSlots > 0) {
          ptx::mbar_wait_warp(&col_full[cs], cphase);
          ctx.col_slot = col_slots + cs * CS::kBytes;
        }
        Epi::tile_begin(ep, rs, shape, ctx, t);
        ptx::mbar_wait_warp(&tmem_full[acc], acc_phase);
        ptx::tc_fence_after_sync();
        const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * kTileN);
#pragma unroll 1
        for (int c = half; c < kTileN / kChunkCols; c += kHalves) {
          uint32_t v[32];
          ptx::tmem_ld_32x32(taddr + (uint32_t)(c * kChunkCols), v);
          ptx::tmem_ld_wait();
          Epi::chunk32(ep, rs, row, t * kTileN + c * kChunkCols, v, shape, ctx);
        }
        ptx::tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(&tmem_empty[acc]);
        if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
        if constexpr (kColSlots > 0) {
          if (lane == 0) ptx::mbar_arrive(&col_empty[cs]);  // (queued entries carry what they need)
          if (++cs == kColSlots) { cs = 0; cphase ^= 1u; }
        }
        Epi::tile_end(ep, rs, shape, ctx);  // work deferred until the accumulator is back with the MMA warp
      }
      Epi::row_end(ep, rs, row, part, shape, ctx);
    }
  }

  ptx::tc_fence_before_sync();
  __syncthreads();
  if (warp_idx == 1) {
    __syncwarp();
    ptx::tc_fence_after_sync();
    ptx::tmem_dealloc<512>(tmem_base);
  }
  release_unit_counter(shape);
}

}  // namespace wealy
