// Epilogue of the symmetric all-vs-all sweep over CLIQUE-SORTED rows (a7, the headline case).
//
// The plan permutes the corpus so that the members of a clique are adjacent ("sorted space").  Then every pair
// that needs an id test -- self, same clique, version-id collision -- lies in a tile next to the diagonal (or
// in one of the handful of tiles a collision pair falls into); the plan marks those tiles `dirty`.  All other
// tiles ("clean", ~99 %) hold negatives only, and scoring an element s = S[row, col] reduces to
//     row direction:  hist[row][#{thr_row < s} - 1] += 1        if s > thr_row[0]
//     col direction:  hist[col][#{thr_col < s} - 1] += 1        if s > thr_col[0]
// with no ids at all.  Because most elements that pass a query's lowest threshold stop at one of the next few
// (the density of negatives falls steeply with s), the lowest kLv thresholds of every query are kept
//   * in registers for the thread's own row,
//   * in a per-tile shared-memory slot for the tile's 256 columns (one 6 KB bulk copy issued by the TMA thread
//     together with the operand tiles; completion on an mbarrier, no CTA barrier per tile),
// and the buckets 0 .. kLv-2 are counted directly (clean tiles: chunk32_clean, counts of compares for the rows and, after
// a transpose of the chunk through shared memory, for the columns; dirty tiles: popc of mask differences for the rows,
// 32x32 bit-matrix transposes + popc for the columns), with one RED per (column, bucket).  Only elements above the kLv-th
// threshold (~1 % of the pairs on SHS100K-shaped data, 7 % pass the first) go through the warp queue, where a
// self-describing entry (value, threshold range, counter index) is binned by a binary search 32 x 2 at a time.
// Dirty tiles apply a validity mask built from the ids (64 shuffles per chunk) and the diagonal test col > row.
//
// Row order inside the sweep: every row / column index in this file is a PLANE row.  The planes, lvl and cinfo store
// each 128-row block of the sorted order with its rows dealt round-robin to the four TMEM lane quadrants
// (spread_sorted_of / spread_plane_of, gemm_core.cuh), because equally hot queries are neighbours in sorted space
// and would otherwise pile up on one pair of epilogue warps.  Ids (s_c, s_i), validity (row < n) and the CSR
// offsets stay in sorted order.
#pragma once
#include "gemm_core.cuh"

namespace wealy {

struct EvalSymParams {
  const float4* lvl;           // [n_col_tiles * 256 (+256)] lowest 4 thresholds of every query, +inf padded
  const uint2* cinfo;          // same length: {CSR offset, number of thresholds}
  const int* s_c;              // [n] clique ids (sorted space)
  const int* s_i;              // [n] version ids
  const float* thr;            // CSR thresholds, ascending per query
  unsigned int* hist;          // CSR rank counters
  const unsigned char* dirty;  // [n_row_blocks][n_col_tiles] tiles that need id tests
  int n_col_tiles;
  int n_row_blocks;            // row blocks of the whole problem (the CTA-pair kernel may be handed one past the end)
  unsigned int total_pairs;
  // top-k in the symmetric sweep (EvalSymEpi<..., kTopk = true>): every query p (plane row) has a static lower bound
  // beta[p] of its k-th best similarity (sampled pre-pass; for the tile's columns it rides in lvl[].w); every
  // candidate above the bound is appended -- row direction and column direction alike -- to the query's list
  // tk_val / tk_idx [p][tk_cap] through the atomic cursor tk_cnt[p] (entries beyond tk_cap are dropped and the
  // finalize kernel reports the query as overflowed).  Candidates are plane rows too.
  const float* beta;
  float* tk_val;
  int* tk_idx;
  int* tk_cnt;
  int tk_cap;
};

__device__ __forceinline__ unsigned bit_transpose32(unsigned x, int lane) {
#pragma unroll
  for (int s = 16; s >= 1; s >>= 1) {
    const unsigned mask = s == 16 ? 0x0000ffffu : s == 8 ? 0x00ff00ffu : s == 4 ? 0x0f0f0f0fu : s == 2 ? 0x33333333u : 0x55555555u;
    const unsigned y = __shfl_xor_sync(0xffffffffu, x, s);
    x = (lane & s) ? ((x & ~mask) | ((y >> s) & mask)) : ((x & mask) | ((y << s) & ~mask));
  }
  return x;
}

template <int kLv, int kQueueCapT = 256, int kCachePairsT = 4096, bool kTopk = false>
struct EvalSymEpi {
  static_assert(kLv >= 2 && kLv <= 4, "2..4 register levels");
  static_assert(!kTopk || kLv <= 3, "the top-k bound of the columns rides in the 4th threshold slot");
  using Params = EvalSymParams;
  static constexpr int kQueueCap = kQueueCapT;
  static constexpr int kCachePairs = kCachePairsT;
  static constexpr unsigned kGlobal = 0x80000000u;
  // per warp: queue of (value, index | kGlobal, range length)
  static constexpr int kOffQx = kQueueCap * 4;
  static constexpr int kOffQn = kOffQx + kQueueCap * 4;
  // + a staging area [16 columns][32 lanes]: the accumulator registers of half a chunk, so that a lane can fetch
  //   the few elements it queues by (dynamic) column index instead of walking all 32 registers under predicates
  static constexpr int kStageCols = 16;
  static constexpr int kOffStage = kOffQn + kQueueCap * 4;
  static constexpr int kWarpScratchBytes = kOffStage + kStageCols * 32 * 4;
  // per CTA: row-block threshold cache, then the ring of per-tile column slots
  static constexpr int kColSlots = 3;
  static constexpr int kLvlBytes = kTileN * 16;
  static constexpr int kInfoBytes = kTileN * 8;
  static constexpr int kColSlotBytes = kLvlBytes + kInfoBytes;
  static constexpr int kOffColSlots = (kCachePairs * 4 + 15) / 16 * 16;
  static constexpr int kCtaScratchBytes = kOffColSlots + kColSlots * kColSlotBytes;

  // what the TMA thread copies into the column slot of tile t
  __device__ static __forceinline__ void col_bulk_src(const Params& p, int t, const void*& s0, const void*& s1) {
    s0 = p.lvl + (size_t)t * kTileN;
    s1 = p.cinfo + (size_t)t * kTileN;
  }

  struct RowState {
    float t[kLv];            // this row's lowest thresholds (+inf beyond its count)
    unsigned rc[kLv - 1];    // direct counters of buckets 0 .. kLv-2 (flushed at the end of the unit)
    unsigned rinfo;          // queue index of this row's deep entries: cache offset + kLv, or kGlobal | (off + kLv)
    int rpc;                 // thresholds beyond the kLv-th
    int qc, qi;
    unsigned off;
    int qn;                  // queued entries (warp-uniform)
    int n_cached;
    unsigned base;           // CSR offset of the unit's first row
    int row_glob, row_ok, dirty;
    float beta;              // kTopk: lower bound of this row's k-th best similarity
  };

  __device__ static __forceinline__ float* q_val(const EpiCtx& c) { return reinterpret_cast<float*>(c.warp_scratch); }
  __device__ static __forceinline__ unsigned* q_idx(const EpiCtx& c) { return reinterpret_cast<unsigned*>(c.warp_scratch + kOffQx); }
  __device__ static __forceinline__ int* q_len(const EpiCtx& c) { return reinterpret_cast<int*>(c.warp_scratch + kOffQn); }
  __device__ static __forceinline__ float* stage(const EpiCtx& c) { return reinterpret_cast<float*>(c.warp_scratch + kOffStage); }
  __device__ static __forceinline__ float* thr_s(const EpiCtx& c) { return reinterpret_cast<float*>(c.cta_scratch); }

  __device__ static __forceinline__ float lvl_of(const float4& v, int j) {
    return j == 0 ? v.x : (j == 1 ? v.y : (j == 2 ? v.z : v.w));
  }

  __device__ static __forceinline__ void row_begin(const Params& p, RowState& st, int row, int part,
                                                   const GemmShape& sh, const EpiCtx& ctx) {
    (void)part;
    const float inf = __int_as_float(0x7f800000);
#pragma unroll
    for (int j = 0; j < kLv; ++j) st.t[j] = inf;
#pragma unroll
    for (int j = 0; j < kLv - 1; ++j) st.rc[j] = 0u;
    st.qc = st.qi = 0;
    st.off = 0u;
    st.beta = inf;
    int cnt = 0;
    // `row` (like every row / column index in here) is a PLANE row: rows are stored in spread order (gemm_core.cuh),
    // lvl / cinfo are indexed the same way; ids and validity go through the sorted index
    const int srow = spread_sorted_of(row);
    st.row_ok = srow < sh.m_rows;
    if (st.row_ok) {
      const float4 v = __ldg(p.lvl + row);
#pragma unroll
      for (int j = 0; j < kLv; ++j) st.t[j] = lvl_of(v, j);
      const uint2 ci = __ldg(p.cinfo + row);
      st.off = ci.x;
      cnt = (int)ci.y;
      st.qc = __ldg(p.s_c + srow);
      st.qi = __ldg(p.s_i + srow);
      if constexpr (kTopk) st.beta = __ldg(p.beta + row);
    }
    st.qn = 0;
    st.row_glob = row;
    st.dirty = 0;
    // cooperative fill of the row block's threshold cache (the previous unit's row_end left it flushed)
    st.base = __ldg(p.cinfo + ctx.row_base).x;
    const unsigned end = (ctx.row_base + ctx.row_span < sh.m_rows) ? __ldg(p.cinfo + ctx.row_base + ctx.row_span).x : p.total_pairs;
    const unsigned total = end - st.base;
    st.n_cached = (int)(total < (unsigned)kCachePairs ? total : (unsigned)kCachePairs);
    float* ts = thr_s(ctx);
    for (int i = ctx.tid; i < st.n_cached; i += ctx.nthreads) ts[i] = __ldg(p.thr + st.base + i);
    const unsigned rel = st.off - st.base;
    const bool cached = st.row_ok && rel + (unsigned)cnt <= (unsigned)st.n_cached;
    st.rinfo = cached ? (rel + kLv) : (kGlobal | (st.off + kLv));
    st.rpc = cnt - kLv;
    ptx::named_barrier_sync(1, ctx.nthreads);
  }

  __device__ static __forceinline__ int warp_incl_scan(int v, int lane) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, v, o);
      if (lane >= o) v += t;
    }
    return v;
  }

  // One queued element: s lies above the kLv lowest thresholds of its query; idx addresses the kLv-th threshold
  // slot + 1 (shared-memory cache offset, or global CSR index with kGlobal), len thresholds remain to search.
  // (kTopk: a queue entry with a NEGATIVE length is a top-k candidate: idx = the query's plane row, -1 - len = the
  //  candidate's plane row; it is appended to the query's list instead of being binned)
  struct Ent {
    float s;
    unsigned idx;
    int len;
    int cand;
    bool on;
    const float* tp;
  };
  __device__ static __forceinline__ void fetch(const Params& p, const EpiCtx& ctx, Ent& en, int r, int end) {
    en.on = r < end;
    en.s = en.on ? q_val(ctx)[r] : 0.f;
    en.idx = en.on ? q_idx(ctx)[r] : 0u;
    const int raw = en.on ? q_len(ctx)[r] : 0;
    en.len = max(raw, 0);
    en.cand = kTopk ? -1 - raw : -1;   // >= 0 for a top-k entry
    en.tp = (en.idx & kGlobal) ? (p.thr + (en.idx & ~kGlobal)) : (thr_s(ctx) + en.idx);
  }
  __device__ static __forceinline__ void count(const Params& p, const RowState& st, const EpiCtx& ctx, const Ent& en,
                                               int lb, int lane) {
    (void)ctx; (void)lane;
    if constexpr (kTopk) {
      if (en.cand >= 0) {
        if (en.on) {
          const int pos = atomicAdd(p.tk_cnt + en.idx, 1);
          if (pos < p.tk_cap) {
            p.tk_val[(size_t)en.idx * p.tk_cap + pos] = en.s;
            p.tk_idx[(size_t)en.idx * p.tk_cap + pos] = en.cand;
          }
        }
        return;
      }
    }
    const bool glob = (en.idx & kGlobal) != 0u;
    // bucket = kLv - 1 + lower bound; cached row entries carry an offset relative to the unit's first row
    const unsigned slot = (en.idx & ~kGlobal) - 1u + (unsigned)lb + (glob ? 0u : st.base);
    if (en.on) atomicAdd(p.hist + slot, 1u);
  }

  // Bin the queued elements: 2 x 32 per iteration so the two dependent load -> compare chains overlap (four chains were
  // measured slower: 23.6 vs 22.7 ms per sweep at C2, 66 vs 48 ms on MAP-0.1 data -- the loop then runs to the depth of
  // the deepest of four searches and the extra registers cost more than the overlap returns).
  __device__ static __forceinline__ void drain(const Params& p, RowState& st, const EpiCtx& ctx) {
    if (st.qn == 0) return;
    const int lane = (int)ptx::lane_id();
    __syncwarp();
    const int end = st.qn;
    for (int r0 = 0; r0 < end; r0 += 64) {
      Ent a, b;
      fetch(p, ctx, a, r0 + lane, end);
      fetch(p, ctx, b, r0 + 32 + lane, end);
      int loa = 0, hia = a.len, lob = 0, hib = b.len;
      while (loa < hia || lob < hib) {
        if (loa < hia) {
          const int mid = (loa + hia) >> 1;
          if (a.tp[mid] < a.s) loa = mid + 1; else hia = mid;
        }
        if (lob < hib) {
          const int mid = (lob + hib) >> 1;
          if (b.tp[mid] < b.s) lob = mid + 1; else hib = mid;
        }
      }
      count(p, st, ctx, a, loa, lane);
      if (r0 + 32 < end) count(p, st, ctx, b, lob, lane);
    }
    __syncwarp();
    st.qn = 0;
  }

  // append the elements selected by the row-direction mask mr and the column-direction mask mcq.  Few bits are set
  // per lane (1.6 % of the pairs are deep), so the registers of half a chunk are parked in shared memory
  // ([column][lane]: conflict free, every lane reads back only its own) and each lane walks its set bits.
  __device__ static __forceinline__ void push(const RowState& st, const EpiCtx& ctx, const uint32_t (&acc)[32], unsigned mr,
                                              unsigned mcq, const uint2* cinf, int pos, unsigned tkr = 0u, unsigned tkc = 0u,
                                              int col0 = 0) {
    float* qv = q_val(ctx);
    unsigned* qx = q_idx(ctx);
    int* ql = q_len(ctx);
    float* stg = stage(ctx) + (ptx::lane_id());
#pragma unroll
    for (int h = 0; h < 32 / kStageCols; ++h) {
      const unsigned sel = ((1u << kStageCols) - 1u) << (h * kStageCols);
      if (!__any_sync(0xffffffffu, ((mr | mcq | tkr | tkc) & sel) != 0u)) continue;
#pragma unroll
      for (int e = 0; e < kStageCols; ++e) stg[e * 32] = __uint_as_float(acc[h * kStageCols + e]);
      unsigned m = mr & sel;
      while (m) {
        const int e = __ffs(m) - 1;
        m &= m - 1;
        qv[pos] = stg[(e - h * kStageCols) * 32];
        qx[pos] = st.rinfo;
        ql[pos] = st.rpc;
        ++pos;
      }
      m = mcq & sel;
      while (m) {
        const int e = __ffs(m) - 1;
        m &= m - 1;
        const uint2 c = cinf[e];
        qv[pos] = stg[(e - h * kStageCols) * 32];
        qx[pos] = kGlobal | (c.x + kLv);
        ql[pos] = (int)c.y - kLv;
        ++pos;
      }
      if constexpr (kTopk) {
        m = tkr & sel;   // this row's candidates: the columns
        while (m) {
          const int e = __ffs(m) - 1;
          m &= m - 1;
          qv[pos] = stg[(e - h * kStageCols) * 32];
          qx[pos] = (unsigned)st.row_glob;
          ql[pos] = -1 - (col0 + e);
          ++pos;
        }
        m = tkc & sel;   // the columns' candidate: this row
        while (m) {
          const int e = __ffs(m) - 1;
          m &= m - 1;
          qv[pos] = stg[(e - h * kStageCols) * 32];
          qx[pos] = (unsigned)(col0 + e);
          ql[pos] = -1 - st.row_glob;
          ++pos;
        }
      }
      __syncwarp();  // (reconverge before the next half overwrites the staging area)
    }
  }

  __device__ static __forceinline__ void tile_begin(const Params& p, RowState& st, const GemmShape& sh,
                                                    const EpiCtx& ctx, int t) {
    (void)sh;
    // (the CTA-pair core draws this CTA's rows from two adjacent row blocks, possibly one past the end)
    st.dirty = 0;
    for (int rbi = ctx.row_base / kTileM; rbi < (ctx.row_base + ctx.row_span) / kTileM; ++rbi)
      st.dirty |= rbi < p.n_row_blocks ? (int)__ldg(p.dirty + (size_t)rbi * p.n_col_tiles + t) : 1;
  }

  // Counting compares.  set.gt.f32.f32 is one FSET writing 1.0f (0x3f800000 = 127 << 23) or 0; summed as INTEGERS,
  // two per IADD3, k of them give 127 k << 23 (mod 2^32), and k < 512 comes back through the inverse of 127 mod 512
  // (383).  The usual (s > t) ? 1 : 0 compiles to FSETP + SEL, one instruction more per compare.
  __device__ static __forceinline__ unsigned gt_one(float a, float b) {
    float r;
    asm("set.gt.f32.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
    return __float_as_uint(r);
  }
  __device__ static __forceinline__ unsigned ones_count(unsigned sum) { return ((sum >> 23) * 383u) & 511u; }
  // m |= bit if a > b: FSETP + a predicated LOP3 (the ternary form compiles to FSETP + SEL + half an IADD3)
  __device__ static __forceinline__ void set_if_gt(unsigned& m, float a, float b, unsigned bit) {
    asm("{\n.reg .pred p;\nsetp.gt.f32 p, %1, %2;\n@p or.b32 %0, %0, %3;\n}" : "+r"(m) : "f"(a), "f"(b), "r"(bit));
  }

  // Clean tile (no ids, no diagonal, no top-k): the same counts as the dense masks of chunk32 with a quarter fewer
  // instructions per element (SASS of EvalSymEpi<4>: about 620 instead of 830 per 32 x 32 chunk, queue excluded).  Both directions rely on the thresholds being ascending (t_j <= t_{j+1}, the
  // K_pos sort), so that an element above level j+1 is above level j too: bucket j holds c_j - c_{j+1} elements,
  // c_j = #{s > t_j}, and levels 0 .. kLv-2 need COUNTS only (gt_one: FSET + half an IADD3 each).  A mask is built for the
  // last level alone (it feeds the queue).
  //   * rows: the thread's row against its thresholds in registers;
  //   * columns: the chunk is transposed through the warp's staging area, 16 columns at a time (lane = column
  //     16 h + lane % 16, rows 16 (lane / 16) .. +16), so that a lane compares against ITS column's thresholds held
  //     in registers -- no broadcast load per element, no bit transposes of the bucket masks.  The two row halves
  //     of a column meet in one shuffle of byte-packed bucket counts; only the last level's mask goes back to the
  //     row layout (one bit transpose) for the queue.
  __device__ static __forceinline__ void chunk32_clean(const Params& p, RowState& st, int col0, const uint32_t (&acc)[32],
                                                       const EpiCtx& ctx, const float4* lv, const uint2* cinf, int lane) {
    constexpr int kCnt = kLv - 1;  // counted levels
    unsigned nr[kCnt];             // c_j of the row, as sums of gt_one
    unsigned dr = 0u;
#pragma unroll
    for (int j = 0; j < kCnt; ++j) nr[j] = 0u;
#pragma unroll
    for (int e = 0; e < 32; ++e) {
      const float s = __uint_as_float(acc[e]);
#pragma unroll
      for (int j = 0; j < kCnt; ++j) nr[j] += gt_one(s, st.t[j]);
      set_if_gt(dr, s, st.t[kCnt], 1u << e);
    }
#pragma unroll
    for (int j = 0; j < kCnt - 1; ++j) st.rc[j] += ones_count(nr[j] - nr[j + 1]);
    st.rc[kCnt - 1] += ones_count(nr[kCnt - 1]) - (unsigned)__popc(dr);

    // columns.  Staging layout of half h: element (row r, column 16 h + e) at e * 32 + (r ^ 4 (e % 8)): the lanes'
    // stores of one column hit 32 banks, and the 16-byte loads of four rows of a column stay contiguous and spread
    // over the banks of each 8-lane phase
    float* stg = stage(ctx);
    const int cc = lane & 15, r0 = lane & 16;
    unsigned cpk = 0u, cdm = 0u;  // lane's column (col0 + lane): bucket counts (one byte per counted level), deep rows
#pragma unroll
    for (int h = 0; h < 2; ++h) {
#pragma unroll
      for (int e = 0; e < 16; ++e) stg[e * 32 + (lane ^ ((e & 7) << 2))] = __uint_as_float(acc[h * 16 + e]);
      __syncwarp();
      const float4 tc = lv[h * 16 + cc];
      const float* src = stg + cc * 32;
      const int sw = (cc & 7) << 2;
      unsigned nc[kCnt];
      unsigned dch = 0u;
#pragma unroll
      for (int j = 0; j < kCnt; ++j) nc[j] = 0u;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float4 q = *reinterpret_cast<const float4*>(src + ((r0 + 4 * k) ^ sw));
        const float v4[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
#pragma unroll
          for (int j = 0; j < kCnt; ++j) nc[j] += gt_one(v4[i], lvl_of(tc, j));
          set_if_gt(dch, v4[i], lvl_of(tc, kCnt), 1u << (4 * k + i));
        }
      }
      __syncwarp();  // (every lane has read the half before the next one, or the queue push, overwrites it)
      unsigned pk = (ones_count(nc[kCnt - 1]) - (unsigned)__popc(dch)) << (8 * (kCnt - 1));
#pragma unroll
      for (int j = 0; j < kCnt - 1; ++j) pk += ones_count(nc[j] - nc[j + 1]) << (8 * j);
      pk += __shfl_xor_sync(0xffffffffu, pk, 16);  // <= 32 per byte
      const unsigned other = __shfl_xor_sync(0xffffffffu, dch, 16);
      if ((lane >> 4) == h) {
        cpk = pk;
        cdm = r0 ? (other | (dch << 16)) : (dch | (other << 16));
      }
    }
    if (cpk != 0u) {
      const unsigned coff = cinf[lane].x;
#pragma unroll
      for (int j = 0; j < kCnt; ++j) {
        const unsigned n = (cpk >> (8 * j)) & 0xffu;
        if (n != 0u) atomicAdd(p.hist + coff + j, n);
      }
    }
    const unsigned dc = __any_sync(0xffffffffu, cdm != 0u) ? bit_transpose32(cdm, lane) : 0u;
    enqueue(p, st, ctx, acc, dr, dc, 0u, 0u, cinf, col0, lane);
  }

  // ---- elements above the kLv-th threshold (and top-k candidates): queue
  __device__ static __forceinline__ void enqueue(const Params& p, RowState& st, const EpiCtx& ctx, const uint32_t (&acc)[32],
                                                 unsigned dr, unsigned dc, unsigned tkr, unsigned tkc, const uint2* cinf,
                                                 int col0, int lane) {
    constexpr unsigned kFull = 0xffffffffu;
    if (!__any_sync(kFull, (dr | dc | tkr | tkc) != 0u)) return;
    const int mine = __popc(dr) + __popc(dc) + __popc(tkr) + __popc(tkc);
    const int incl = warp_incl_scan(mine, lane);
    const int total = __shfl_sync(kFull, incl, 31);
    if (st.qn + total > kQueueCap) drain(p, st, ctx);
    if (total <= kQueueCap) {
      push(st, ctx, acc, dr, dc, cinf, st.qn + incl - mine, tkr, tkc, col0);
      st.qn += total;
    } else {
      // a chunk denser than the whole queue: kQueueCap / 64 columns (<= kQueueCap entries) at a time
      constexpr int kBatchCols = kQueueCap / (kTopk ? 128 : 64);
      static_assert(kBatchCols >= 1 && 32 % kBatchCols == 0, "queue capacity: 64 (128 with top-k) .. 2048, a power of two");
#pragma unroll 1
      for (int g = 0; g < 32 / kBatchCols; ++g) {
        const unsigned sel = ((1u << kBatchCols) - 1u) << (kBatchCols * g);
        const int mine_g = __popc(dr & sel) + __popc(dc & sel) + __popc(tkr & sel) + __popc(tkc & sel);
        const int incl_g = warp_incl_scan(mine_g, lane);
        push(st, ctx, acc, dr & sel, dc & sel, cinf, incl_g - mine_g, tkr & sel, tkc & sel, col0);
        st.qn = __shfl_sync(kFull, incl_g, 31);
        drain(p, st, ctx);
      }
    }
  }

  __device__ static __forceinline__ void chunk32(const Params& p, RowState& st, int row, int col0,
                                                 const uint32_t (&acc)[32], const GemmShape& sh, const EpiCtx& ctx) {
    constexpr unsigned kFull = 0xffffffffu;
    const int lane = (int)ptx::lane_id();
    (void)row;
    const float4* lv = reinterpret_cast<const float4*>(ctx.col_slot) + (col0 & (kTileN - 1));
    const uint2* cinf = reinterpret_cast<const uint2*>(ctx.col_slot + kLvlBytes) + (col0 & (kTileN - 1));
    if constexpr (!kTopk) {
      if (!st.dirty) {
        chunk32_clean(p, st, col0, acc, ctx, lv, cinf, lane);
        return;
      }
    }

    unsigned m[kLv], mc[kLv];
    unsigned tkr = 0u, tkc = 0u;  // kTopk: elements above the row's / the column's top-k bound
#pragma unroll
    for (int j = 0; j < kLv; ++j) m[j] = mc[j] = 0u;
#pragma unroll
    for (int e = 0; e < 32; ++e) {
      const float s = __uint_as_float(acc[e]);
      const float4 c = lv[e];  // broadcast load: the column's lowest thresholds
#pragma unroll
      for (int j = 0; j < kLv; ++j) {
        m[j] |= (s > st.t[j]) ? (1u << e) : 0u;
        mc[j] |= (s > lvl_of(c, j)) ? (1u << e) : 0u;
      }
      if constexpr (kTopk) {
        tkr |= (s > st.beta) ? (1u << e) : 0u;
        tkc |= (s > c.w) ? (1u << e) : 0u;
      }
    }
    if (st.dirty) {
      // tile with self / same-clique / colliding pairs, or ragged edges: candidates by id, above the diagonal only
      const int scol = spread_sorted_of(col0 + lane);
      const bool ok = scol < sh.n_cols;
      const int cc = ok ? __ldg(p.s_c + scol) : 0;
      const int ci = ok ? __ldg(p.s_i + scol) : 0;
      unsigned valid = 0u, validk = 0u;  // negatives for the rank counts / top-k candidates (a relevant item is one)
#pragma unroll
      for (int e = 0; e < 32; ++e) {
        const int cce = __shfl_sync(kFull, cc, e);
        const int cie = __shfl_sync(kFull, ci, e);
        const int oke = __shfl_sync(kFull, (int)ok, e);
        valid |= (oke && cce != st.qc && cie != st.qi) ? (1u << e) : 0u;
        if constexpr (kTopk) validk |= (oke && cie != st.qi) ? (1u << e) : 0u;
      }
      const int d = st.row_glob - col0;  // columns 0..d of this chunk are on or below the diagonal
      const unsigned above = d < 0 ? 0xffffffffu : (d >= 31 ? 0u : (0xffffffffu << (d + 1)));
      valid &= above;
      validk &= above;
      if (!st.row_ok) valid = validk = 0u;
#pragma unroll
      for (int j = 0; j < kLv; ++j) {
        m[j] &= valid;
        mc[j] &= valid;
      }
      tkr &= validk;
      tkc &= validk;
    }
    if constexpr (kTopk) {
      if (!__any_sync(kFull, (m[0] | mc[0] | tkr | tkc) != 0u)) return;
    } else {
      if (!__any_sync(kFull, (m[0] | mc[0]) != 0u)) return;
    }

    // ---- buckets 0 .. kLv-2, counted directly
#pragma unroll
    for (int j = 0; j < kLv - 1; ++j) st.rc[j] += (unsigned)__popc(m[j] ^ m[j + 1]);
    if (__any_sync(kFull, (mc[0] ^ mc[kLv - 1]) != 0u)) {
      const unsigned coff = cinf[lane].x;
#pragma unroll
      for (int j = 0; j < kLv - 1; ++j) {
        const unsigned n = (unsigned)__popc(bit_transpose32(mc[j] ^ mc[j + 1], lane));  // rows in bucket j of column `lane`
        if (n != 0u) atomicAdd(p.hist + coff + j, n);
      }
    }

    enqueue(p, st, ctx, acc, m[kLv - 1], mc[kLv - 1], tkr, tkc, cinf, col0, lane);
  }

  __device__ static __forceinline__ void tile_end(const Params& p, RowState& st, const GemmShape&, const EpiCtx& ctx) {
    // the accumulator is back with the MMA warp: bin what has piled up (full rounds keep every lane busy)
    if (st.qn >= kQueueCap / 2) drain(p, st, ctx);
  }

  __device__ static __forceinline__ void row_end(const Params& p, RowState& st, int row, int part,
                                                 const GemmShape& sh, const EpiCtx& ctx) {
    (void)row; (void)part; (void)sh;
    drain(p, st, ctx);
    if (st.row_ok) {
#pragma unroll
      for (int j = 0; j < kLv - 1; ++j)
        if (st.rc[j] != 0u) atomicAdd(p.hist + st.off + j, st.rc[j]);
    }
    ptx::named_barrier_sync(1, ctx.nthreads);  // every warp is done with the threshold cache before the next unit refills it
  }
};

}  // namespace wealy
