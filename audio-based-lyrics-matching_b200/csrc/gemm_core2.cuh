// CTA-pair variant of the contraction core (gemm_core.cuh) for the symmetric evaluation sweep: two CTAs of a
// cluster (two SMs of one TPC) work on one 256 x 256 tile with tcgen05.mma.cta_group::2.
//
//   * each CTA owns 128 rows of the tile -- the even (rank 0) or odd (rank 1) rows of the 256-row "super" row block
//     S, loaded with row-strided TMA boxes -- and keeps the accumulator of those rows in its own TMEM.  The two
//     epilogues are coupled through the shared accumulator hand-over (the pair advances at the pace of the slower
//     one), and the data-dependent epilogue work is a property of the rows (neighbouring rows belong to the same
//     clique): interleaving splits it evenly between the two CTAs;
//   * each CTA loads its 128 A rows and only HALF of the tile's 256 B rows (columns 128 cta_rank .. +128); the
//     tensor cores of both SMs read the two halves from both shared memories.  Per tile the pair moves
//     2 x (A + B/2) instead of 2 x (A + B) through L2 -> shared memory, and a pipeline stage is 32 KB instead of
//     48 KB (4 stages instead of 3 next to the same epilogue scratch);
//   * the leader CTA (rank 0) issues the MMAs; TMA completions of both CTAs are counted on the leader's `full`
//     barriers (cp.async.bulk.tensor.cta_group::2), tcgen05.commit multicasts to the `empty` / `tmem_full`
//     barriers of both CTAs, the epilogue warps of both CTAs arrive on the leader's `tmem_empty`;
//   * units are (super row block) x (chunk of column tiles), handed out dynamically by the leader's TMA thread,
//     which publishes the unit index into the mailboxes of both CTAs (st.shared::cluster + remote mbarrier arrive);
//   * kDynChunks (every epilogue with per-tile column slots, i.e. the symmetric evaluation's EvalSymEpi): the epilogue
//     warps of a TMEM lane quadrant do not own fixed 32-column chunks of a tile; they CLAIM the chunks of the unit's
//     tiles one by one from a shared-memory counter (chunk stream g -> tile g / 8, chunk g % 8).  The rows of a
//     quadrant are the same for all its warps, so any of them can score any chunk; a warp held up by a hot chunk
//     (deep queue, dirty tile) simply claims fewer, and a fast one runs ahead into the next tile as soon as its
//     accumulator is ready.  The accumulator hand-over then waits for the SUM of the warps' work, not for the
//     slowest warp of 2 x kEpiWarps: every chunk arrives on `tmem_empty` on its own.
#pragma once
#include "gemm_core.cuh"

namespace wealy {

template <int kPasses, int kBlockK, int kStages>
struct PairSmem {
  static constexpr int kSwizzle = kBlockK * 2;
  static constexpr int kTileBytes = kTileM * kBlockK * 2;  // 128 rows of one plane (A rows, or half of the B rows)
  static constexpr int kPlanes = kPasses == 3 ? 2 : 1;
  static constexpr int kStageBytes = kPlanes * 2 * kTileBytes;
  static constexpr int kBarBytes = 512;
  static constexpr int kCore = kStages * kStageBytes + kBarBytes;
  static constexpr int total(int epi_warps, int scratch_per_warp, int cta_scratch) {
    return kCore + epi_warps * scratch_per_warp + cta_scratch + 1024;
  }
};

template <class Epi, int kPasses, int kBlockK, int kEpiWarps, int kStages>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(64 + kEpiWarps * 32, 1)
gemm_pair_kernel(const __grid_constant__ GemmTmaps tmaps, const GemmShape shape, const typename Epi::Params ep) {
  using SM = PairSmem<kPasses, kBlockK, kStages>;
  using CS = ColSlotTraits<Epi>;
  constexpr int kHalves = kEpiWarps / 4;
  constexpr int kColSlots = CS::kSlots;
  constexpr bool kDynChunks = kColSlots > 0;  // dynamic chunk claiming; the other epilogues own fixed chunks
  static_assert(kEpiWarps == 8 || kEpiWarps == 12, "8 or 12 epilogue warps (2 or 3 per TMEM lane quadrant)");
  static_assert(kTileN == 2 * kTileM, "symmetric tile range assumes 256-wide column tiles over 256-row super blocks");

  extern __shared__ uint8_t smem_raw[];
  // (the dynamic shared memory of both CTAs starts at the same offset, so the aligned layouts coincide)
  uint8_t* smem = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* bar_base = smem + kStages * SM::kStageBytes;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(bar_base);  // used in the leader only
  uint64_t* empty_bar = full_bar + kStages;
  uint64_t* tmem_full = empty_bar + kStages;
  uint64_t* tmem_empty = tmem_full + 2;                        // leader only: both CTAs' epilogue warps arrive
  uint64_t* unit_full = tmem_empty + 2;
  uint64_t* unit_empty = unit_full + 2;                        // leader only
  uint64_t* col_full = unit_empty + 2;
  uint64_t* col_empty = col_full + (kColSlots > 0 ? kColSlots : 1);
  int* unit_slot = reinterpret_cast<int*>(col_empty + (kColSlots > 0 ? kColSlots : 1));
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(unit_slot + 2);
  int* chunk_ctr = reinterpret_cast<int*>(tmem_slot + 2);      // [2 unit slots][4 quadrants] chunk claim counters
  static_assert((2 * kStages + 8 + 2 * (kColSlots > 0 ? kColSlots : 1)) * 8 + 16 + 32 <= SM::kBarBytes, "barrier area");
  constexpr int kChunksPerTile = kTileN / kChunkCols;          // per quadrant
  uint8_t* scratch_base = bar_base + SM::kBarBytes;
  uint8_t* col_slots = scratch_base + kEpiWarps * Epi::kWarpScratchBytes + CS::kOffset;

  const int warp_idx = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const int lane = (int)ptx::lane_id();
  const uint32_t cta_rank = ptx::cluster_ctarank();
  const bool leader = cta_rank == 0;

  if (warp_idx == 0 && lane == 0) {
    ptx::prefetch_tensormap(&tmaps.a_hi);
    ptx::prefetch_tensormap(&tmaps.b_hi);
    if (kPasses == 3) {
      ptx::prefetch_tensormap(&tmaps.a_lo);
      ptx::prefetch_tensormap(&tmaps.b_lo);
    }
    for (int s = 0; s < kStages; ++s) {
      ptx::mbar_init(&full_bar[s], 1);   // the leader's producer arrives once, with the bytes of both CTAs
      ptx::mbar_init(&empty_bar[s], 1);  // one multicast commit
    }
    for (int a = 0; a < 2; ++a) {
      ptx::mbar_init(&tmem_full[a], 1);
      ptx::mbar_init(&tmem_empty[a], kDynChunks ? 2 * 4 * kChunksPerTile : 2 * kEpiWarps);  // per chunk / per warp
      ptx::mbar_init(&unit_full[a], 1);
      ptx::mbar_init(&unit_empty[a], 2 * kEpiWarps + 2);  // leader: MMA thread + epilogue warps; peer: TMA thread + epilogue warps
    }
    for (int c = 0; c < kColSlots; ++c) {
      ptx::mbar_init(&col_full[c], 1);
      ptx::mbar_init(&col_empty[c], 4 * kChunksPerTile);  // per claimed chunk
    }
    for (int k = 0; k < 8; ++k) chunk_ctr[k] = 0;
    ptx::fence_mbar_init();
  }
  if (warp_idx == 1) ptx::tmem_alloc_pair<512>(tmem_slot);
  ptx::tc_fence_before_sync();
  ptx::cluster_sync_all();
  ptx::tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;

  const int n_units = shape.n_row_blocks * shape.n_col_chunks;  // n_row_blocks counts SUPER row blocks here

  // unit -> (chunk, super row block S); symmetric sweeps: rows [256 S, 256 S + 256) need column tiles >= S
  auto unit_tiles_c = [&](int u, int& S, int& t0, int& t1, int& chunk) {
    decode_unit(shape, u, chunk, S);
    t1 = min((chunk + 1) * shape.tiles_per_chunk, shape.n_col_tiles);
    t0 = shape.sym ? max(chunk * shape.tiles_per_chunk, S) : chunk * shape.tiles_per_chunk;
  };
  auto unit_tiles = [&](int u, int& S, int& t0, int& t1) {
    int chunk;
    unit_tiles_c(u, S, t0, t1, chunk);
  };

  if (warp_idx == 0) {
    // ===================================================== TMA producer (one thread per CTA)
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      int us = 0;
      uint32_t uphase = 0;
      int cs = 0;
      uint32_t cphase = 0;
      const uint32_t leader_full0 = ptx::map_to_cta(&full_bar[0], 0);
      const uint32_t peer_unit_full0 = ptx::map_to_cta(&unit_full[0], 1);
      const uint32_t peer_unit_slot0 = ptx::map_to_cta(&unit_slot[0], 1);
      const uint32_t leader_unit_empty0 = ptx::map_to_cta(&unit_empty[0], 0);
      const uint32_t peer_chunk_ctr0 = ptx::map_to_cta(&chunk_ctr[0], 1);
      while (true) {
        int u;
        if (leader) {
          // fetch the next unit and publish it to the consumers of both CTAs
          ptx::mbar_wait_cluster(&unit_empty[us], uphase ^ 1u);
          u = atomicAdd(shape.unit_counter, 1);
          if (u >= n_units) u = -1;
          unit_slot[us] = u;
          ptx::st_cluster_u32(peer_unit_slot0 + 4u * us, (uint32_t)u);
          if constexpr (kDynChunks) {
            // (every consumer of the slot's previous unit has arrived on unit_empty: nobody claims from these any more)
            for (int k = 0; k < 4; ++k) {
              chunk_ctr[us * 4 + k] = 0;
              ptx::st_cluster_u32(peer_chunk_ctr0 + 4u * (us * 4 + k), 0u);
            }
          }
          ptx::mbar_arrive(&unit_full[us]);
          ptx::mbar_arrive_cluster(peer_unit_full0 + 8u * us);  // release.cluster: orders the slot write before it
        } else {
          ptx::mbar_wait_cluster(&unit_full[us], uphase);
          u = unit_slot[us];
          ptx::mbar_arrive_cluster_relaxed(leader_unit_empty0 + 8u * us);
        }
        if (++us == 2) { us = 0; uphase ^= 1u; }
        if (u < 0) break;
        int rb, t0, t1;
        unit_tiles(u, rb, t0, t1);
        for (int t = t0; t < t1; ++t) {
          if constexpr (kColSlots > 0) {
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
            ptx::mbar_wait_cluster(&empty_bar[stage], phase ^ 1u);
            uint8_t* st = smem + stage * SM::kStageBytes;
            if (leader) ptx::mbar_expect_tx(&full_bar[stage], 2 * SM::kStageBytes);
            const uint32_t fb = leader_full0 + 8u * stage;
            const int brow = t * kTileN + (int)cta_rank * kTileM;  // this CTA's half of the tile's candidate rows
            // layout of a stage: A_hi | A_lo | B_hi(half) | B_lo(half)   (single pass: A_hi | B_hi)
            // interleaved: every second row of the super block (rb), this rank's parity; else this rank's half
            const int arow = (shape.sym & 2) ? rb * 2 * kTileM + (int)cta_rank : rb * 2 * kTileM + (int)cta_rank * kTileM;
            ptx::tma_load_2d_pair(st, &tmaps.a_hi, fb, kb * kBlockK, arow, ptx::kEvictLast);
            ptx::tma_load_2d_pair(st + SM::kPlanes * SM::kTileBytes, &tmaps.b_hi, fb, kb * kBlockK, brow, ptx::kEvictNormal);
            if (kPasses == 3) {
              ptx::tma_load_2d_pair(st + SM::kTileBytes, &tmaps.a_lo, fb, kb * kBlockK, arow, ptx::kEvictLast);
              ptx::tma_load_2d_pair(st + 3 * SM::kTileBytes, &tmaps.b_lo, fb, kb * kBlockK, brow, ptx::kEvictNormal);
            }
            if (++stage == kStages) { stage = 0; phase ^= 1u; }
          }
        }
      }
    }
  } else if (warp_idx == 1) {
    // ===================================================== MMA issuer (one thread of the leader CTA)
    if (lane == 0 && leader) {
      constexpr uint32_t idesc = ptx::make_idesc_f16(2 * kTileM, kTileN, false);  // M = 256 over the pair
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      int us = 0;
      uint32_t uphase = 0;
#ifdef WEALY_PROFILE_WAITS
      // where the MMA thread waits (diagnostic build: -DWEALY_PROFILE_WAITS, printed by a few CTAs)
      long long w_unit = 0, w_acc = 0, w_full = 0, n_tiles_done = 0;
      const long long t_begin = clock64();
#define WEALY_TIMED(var, stmt) { const long long _t = clock64(); stmt; var += clock64() - _t; }
#else
#define WEALY_TIMED(var, stmt) stmt;
#endif
      while (true) {
        WEALY_TIMED(w_unit, ptx::mbar_wait(&unit_full[us], uphase))
        const int u = unit_slot[us];
        ptx::mbar_arrive(&unit_empty[us]);
        if (++us == 2) { us = 0; uphase ^= 1u; }
        if (u < 0) break;
        int rb, t0, t1;
        unit_tiles(u, rb, t0, t1);
        for (int t = t0; t < t1; ++t) {
          WEALY_TIMED(w_acc, ptx::mbar_wait_cluster(&tmem_empty[acc], acc_phase ^ 1u))  // both CTAs' epilogues have drained this accumulator
          ptx::tc_fence_after_sync();
#ifdef WEALY_PROFILE_WAITS
          ++n_tiles_done;
#endif
          const uint32_t d_tmem = tmem_base + (uint32_t)(acc * kTileN);
          for (int kb = 0; kb < shape.k_blocks; ++kb) {
            WEALY_TIMED(w_full, ptx::mbar_wait_cluster(&full_bar[stage], phase))
            ptx::tc_fence_after_sync();
            const uint32_t st = ptx::smem_u32(smem + stage * SM::kStageBytes);
            const uint64_t a_hi = ptx::make_smem_desc<SM::kSwizzle>(st);
            const uint64_t a_lo = ptx::make_smem_desc<SM::kSwizzle>(st + SM::kTileBytes);
            const uint64_t b_hi = ptx::make_smem_desc<SM::kSwizzle>(st + SM::kPlanes * SM::kTileBytes);
            const uint64_t b_lo = ptx::make_smem_desc<SM::kSwizzle>(st + 3 * SM::kTileBytes);
#pragma unroll
            for (int kk = 0; kk < kBlockK / kUmmaK; ++kk) {
              const uint64_t adv = (uint64_t)((kk * kUmmaK * 2) >> 4);
              ptx::umma_f16_pair(d_tmem, a_hi + adv, b_hi + adv, idesc, (uint32_t)((kb | kk) != 0));
              if (kPasses == 3) {
                ptx::umma_f16_pair(d_tmem, a_hi + adv, b_lo + adv, idesc, 1u);
                ptx::umma_f16_pair(d_tmem, a_lo + adv, b_hi + adv, idesc, 1u);
              }
            }
            ptx::umma_commit_pair(&empty_bar[stage]);  // both CTAs' slots are reusable once these MMAs retire
            if (kb == shape.k_blocks - 1) ptx::umma_commit_pair(&tmem_full[acc]);
            if (++stage == kStages) { stage = 0; phase ^= 1u; }
          }
          if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
        }
      }
#ifdef WEALY_PROFILE_WAITS
      if ((blockIdx.x % 37) == 0)
        printf("wealy waits: cta %d tiles %lld total %lld cyc | wait unit %lld acc(epilogue) %lld full(tma) %lld\n", (int)blockIdx.x,
               n_tiles_done, clock64() - t_begin, w_unit, w_acc, w_full);
#endif
    }
  } else {
    // ===================================================== epilogue warps (both CTAs)
    const int ew = warp_idx - 2;
    const int quad = warp_idx & 3;
    const int half = ew >> 2;
    const int row_in_tile = quad * 32 + lane;
    int acc = 0;
    uint32_t acc_phase = 0;
    int us = 0;
    uint32_t uphase = 0;
    const uint32_t leader_unit_empty0 = ptx::map_to_cta(&unit_empty[0], 0);
    const uint32_t leader_tmem_empty0 = ptx::map_to_cta(&tmem_empty[0], 0);
    unsigned tile_seq = 0;  // kDynChunks: tiles this CTA has been through (every role counts the same)
    int pending_slot = -1;  // kDynChunks: unit slot whose release is deferred until the unit's chunks are all claimed
    while (true) {
      ptx::mbar_wait_cluster_warp(&unit_full[us], uphase);
      const int u = unit_slot[us];
      const int us_claim = us;
      __syncwarp();
      if constexpr (kDynChunks) {
        // the slot's claim counters stay in use for the whole unit: release the PREVIOUS unit's slot now, this one
        // after its last chunk has been claimed (2-deep mailbox: the producer is then at most one unit ahead)
        if (pending_slot >= 0 && lane == 0) ptx::mbar_arrive_cluster_relaxed(leader_unit_empty0 + 8u * pending_slot);
        pending_slot = us;
      } else {
        if (lane == 0) ptx::mbar_arrive_cluster_relaxed(leader_unit_empty0 + 8u * us);
      }
      if (++us == 2) { us = 0; uphase ^= 1u; }
      if (u < 0) break;
      int rb, t0, t1, chunk;
      unit_tiles_c(u, rb, t0, t1, chunk);
      if (t0 >= t1) continue;
      const int row = (shape.sym & 2) ? rb * 2 * kTileM + 2 * row_in_tile + (int)cta_rank  // rb is the SUPER row block here
                                      : rb * 2 * kTileM + (int)cta_rank * kTileM + row_in_tile;
      const int part = chunk * kHalves + half;  // partial-result slot of epilogues that keep per-(chunk, warp) state
      typename Epi::RowState rs;
      EpiCtx ctx;
      ctx.warp_scratch = scratch_base + ew * Epi::kWarpScratchBytes;
      ctx.cta_scratch = scratch_base + kEpiWarps * Epi::kWarpScratchBytes;
      ctx.tid = ew * 32 + lane;
      ctx.nthreads = kEpiWarps * 32;
      // interleaved rows: the pair's 256-row super block (the CTAs' rows alternate); otherwise this CTA's own 128 rows
      ctx.row_base = (shape.sym & 2) ? rb * 2 * kTileM : rb * 2 * kTileM + (int)cta_rank * kTileM;
      ctx.row_span = (shape.sym & 2) ? 2 * kTileM : kTileM;
      ctx.first_col = t0 * kTileN + half * kChunkCols;
      ctx.col_step = kHalves * kChunkCols;
      ctx.col_slot = nullptr;
      Epi::row_begin(ep, rs, row, part, shape, ctx);
      if constexpr (kDynChunks) {
        // chunk stream of this quadrant: g -> (tile g / 8, chunk g % 8); tiles are numbered through the CTA's
        // lifetime (tile_seq) so that barrier slots and phases follow from the number alone
        const int n_tiles = t1 - t0;
        const int total = n_tiles * kChunksPerTile;
        int* ctr = &chunk_ctr[us_claim * 4 + quad];
        int cur = -1, a_cur = 0, c_cur = 0;
        while (true) {
          int g = 0;
          if (lane == 0) g = atomicAdd(ctr, 1);
          g = __shfl_sync(0xffffffffu, g, 0);
          if (g >= total) break;
          const int tile = g / kChunksPerTile, c = g - tile * kChunksPerTile;
          if (tile != cur) {
            if (cur >= 0) Epi::tile_end(ep, rs, shape, ctx);
            const unsigned seq = tile_seq + (unsigned)tile;
            a_cur = (int)(seq & 1u);
            c_cur = (int)(seq % (unsigned)kColSlots);
            ptx::mbar_wait_warp(&col_full[c_cur], (seq / (unsigned)kColSlots) & 1u);
            ctx.col_slot = col_slots + c_cur * CS::kBytes;
            Epi::tile_begin(ep, rs, shape, ctx, t0 + tile);
            ptx::mbar_wait_cluster_warp(&tmem_full[a_cur], (seq >> 1) & 1u);
            ptx::tc_fence_after_sync();
            cur = tile;
          }
          const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(a_cur * kTileN);
          uint32_t v[32];
          ptx::tmem_ld_32x32(taddr + (uint32_t)(c * kChunkCols), v);
          ptx::tmem_ld_wait();
          // the chunk now lives in registers: hand its part of the accumulator back BEFORE scoring it, so that a slow
          // chunk (queue drain, dirty tile) never holds up the tensor pipe; only the column slot stays in use
          ptx::tc_fence_before_sync();
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive_cluster_relaxed(leader_tmem_empty0 + 8u * a_cur);
          Epi::chunk32(ep, rs, row, (t0 + tile) * kTileN + c * kChunkCols, v, shape, ctx);
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(&col_empty[c_cur]);
        }
        if (cur >= 0) Epi::tile_end(ep, rs, shape, ctx);
        tile_seq += (unsigned)n_tiles;
      } else {
      for (int t = t0; t < t1; ++t) {
        Epi::tile_begin(ep, rs, shape, ctx, t);
        ptx::mbar_wait_cluster_warp(&tmem_full[acc], acc_phase);
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
        if (lane == 0) ptx::mbar_arrive_cluster_relaxed(leader_tmem_empty0 + 8u * acc);
        if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
        Epi::tile_end(ep, rs, shape, ctx);
      }
      }
      Epi::row_end(ep, rs, row, part, shape, ctx);
    }
  }

  ptx::tc_fence_before_sync();
  ptx::cluster_sync_all();  // nobody leaves (or frees TMEM) while the peer may still signal or read
  if (warp_idx == 1) {
    ptx::tc_fence_after_sync();
    ptx::tmem_dealloc_pair<512>(tmem_base);
  }
  release_unit_counter(shape);
}

}  // namespace wealy
