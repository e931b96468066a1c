// C-ABI entry points (include/wealy_b200.h) and host-side launch logic.
#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <mutex>
#include <vector>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/iterator/transform_input_iterator.cuh>

#include "../../include/wealy_b200.h"
#include "epilogues.cuh"
#include "eval_sym_epilogue.cuh"
#include "gemm_core2.cuh"
#include "eval_kernels.cuh"
#include "f64_kernels.cuh"
#include "loss_kernels.cuh"
#include "masked_kernels.cuh"
#include "pool_kernels.cuh"
#include "prep.cuh"
#include "redux_kernels.cuh"
#include "topk_sym_kernels.cuh"

using namespace wealy;

// ------------------------------------------------------------------------------------------
// error plumbing
// ------------------------------------------------------------------------------------------
static thread_local char g_err[1024] = "";

static int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

#define CU_TRY(expr)                                                                                     \
  do {                                                                                                   \
    cudaError_t _e = (expr);                                                                             \
    if (_e != cudaSuccess) return fail(WEALY_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), \
                                       __FILE__, __LINE__);                                              \
  } while (0)

#define W_TRY(expr)            \
  do {                         \
    int _s = (expr);           \
    if (_s != WEALY_OK) return _s; \
  } while (0)

extern "C" const char* wealy_last_error(void) { return g_err; }
extern "C" int wealy_version(void) { return 100; }

static inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }
static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

static int env_int(const char* name, int dflt) {
  const char* v = getenv(name);
  return v ? atoi(v) : dflt;
}

static int num_sms() {
  static int cached = 0;
  if (!cached) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&cached, cudaDevAttrMultiProcessorCount, dev);
    if (cached <= 0) cached = 148;
  }
  return cached;
}

// Stream-ordered device allocations from a PRIVATE memory pool per device (the process-wide default pool and
// torch's caching allocator are left alone).  Freed blocks stay cached in the pool so that an evaluation plan
// rebuilt on every call (the end-to-end path of bench.py) costs no cudaMalloc / cudaFree round trips through the
// driver; wealy_eval_plan_destroy trims the pool back to WEALY_POOL_KEEP_MB (default 4096) so that a training
// process that evaluates now and then does not sit on the plan scratch for ever.
static cudaMemPool_t g_pools[64] = {nullptr};

static cudaMemPool_t device_pool(int dev) {
  if (dev < 0 || dev >= 64) return nullptr;
  if (!g_pools[dev]) {
    cudaMemPoolProps props;
    memset(&props, 0, sizeof(props));
    props.allocType = cudaMemAllocationTypePinned;
    props.handleTypes = cudaMemHandleTypeNone;
    props.location.type = cudaMemLocationTypeDevice;
    props.location.id = dev;
    cudaMemPool_t pool = nullptr;
    if (cudaMemPoolCreate(&pool, &props) != cudaSuccess) {
      cudaGetLastError();
      return nullptr;
    }
    unsigned long long keep = ~0ull;  // bounded by the explicit trim below, not by every stream synchronisation
    cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    g_pools[dev] = pool;
  }
  return g_pools[dev];
}

static cudaError_t dev_alloc(void** ptr, size_t bytes, cudaStream_t s) {
  int dev = 0;
  cudaGetDevice(&dev);
  cudaMemPool_t pool = device_pool(dev);
  if (pool) return cudaMallocFromPoolAsync(ptr, bytes, pool, s);
  return cudaMallocAsync(ptr, bytes, s);
}
static void dev_free(void* ptr, cudaStream_t s) {
  if (ptr) cudaFreeAsync(ptr, s);
}
// The large buffers of a plan (operand planes, top-k candidate lists) additionally go through a small free list of whole
// blocks.  A serving loop destroys and creates a plan per request; handing the freed 0.4 GB block of one plan straight
// to the next keeps the driver's pool out of that rhythm -- its stream-ordered sub-allocator was measured to stall
// cudaMallocFromPoolAsync for 20-400 ms now and then when a block of that size had to be found while other work was
// in flight (profiles/r02_summary.md, "EvalPipeline").  A block is reused on any stream: the new owner's stream waits
// for the event recorded where the old owner released it.
struct BigBlock {
  void* ptr;
  size_t bytes;
  int dev;
  cudaStream_t stream;
  cudaEvent_t released;
};
static std::mutex g_big_mu;
static std::vector<BigBlock> g_big;
static const size_t kBigMin = (size_t)32 << 20;

static cudaError_t big_alloc(void** ptr, size_t* cap, size_t bytes, cudaStream_t s) {
  *ptr = nullptr;
  *cap = 0;
  int dev = 0;
  cudaGetDevice(&dev);
  if (bytes >= kBigMin) {
    std::lock_guard<std::mutex> lock(g_big_mu);
    int best = -1;
    for (int k = 0; k < (int)g_big.size(); ++k) {
      const BigBlock& b = g_big[k];
      // (a block up to 1.5x the request: the next request of the same workload fits exactly, a much smaller one
      //  should not pin a large block)
      if (b.dev == dev && b.bytes >= bytes && b.bytes <= bytes + bytes / 2 && (best < 0 || b.bytes < g_big[best].bytes)) best = k;
    }
    if (best >= 0) {
      BigBlock b = g_big[best];
      g_big.erase(g_big.begin() + best);
      if (b.stream != s) cudaStreamWaitEvent(s, b.released, 0);
      cudaEventDestroy(b.released);
      *ptr = b.ptr;
      *cap = b.bytes;
      return cudaSuccess;
    }
  }
  cudaError_t e = dev_alloc(ptr, bytes, s);
  if (e == cudaErrorMemoryAllocation) {
    // out of memory with blocks parked: give them back to the pool (and the pool's idle pages to the driver), retry once
    cudaGetLastError();
    {
      std::lock_guard<std::mutex> lock(g_big_mu);
      for (size_t k = 0; k < g_big.size();) {
        if (g_big[k].dev != dev) { ++k; continue; }
        cudaFreeAsync(g_big[k].ptr, g_big[k].stream);
        cudaEventDestroy(g_big[k].released);
        g_big.erase(g_big.begin() + k);
      }
    }
    cudaDeviceSynchronize();
    e = dev_alloc(ptr, bytes, s);
  }
  if (e == cudaSuccess) *cap = bytes;
  return e;
}
static void big_free(void* ptr, size_t bytes, cudaStream_t s) {
  if (!ptr) return;
  int dev = 0;
  cudaGetDevice(&dev);
  const size_t keep = (size_t)env_int("WEALY_POOL_KEEP_MB", 4096) << 20;
  BigBlock b{ptr, bytes, dev, s, nullptr};
  bool cache = bytes >= kBigMin && bytes <= keep;
  if (cache && (cudaEventCreateWithFlags(&b.released, cudaEventDisableTiming) != cudaSuccess ||
                cudaEventRecord(b.released, s) != cudaSuccess)) {
    cudaGetLastError();
    if (b.released) cudaEventDestroy(b.released);
    cache = false;
  }
  if (!cache) dev_free(ptr, s);
  std::lock_guard<std::mutex> lock(g_big_mu);
  if (cache) g_big.push_back(b);
  // oldest blocks go back to the pool once the list holds more than the limit
  size_t total = 0;
  for (const BigBlock& x : g_big) total += x.dev == dev ? x.bytes : 0;
  for (size_t k = 0; k < g_big.size() && total > keep;) {
    if (g_big[k].dev != dev) { ++k; continue; }
    total -= g_big[k].bytes;
    cudaFreeAsync(g_big[k].ptr, g_big[k].stream);
    cudaEventDestroy(g_big[k].released);
    g_big.erase(g_big.begin() + k);
  }
}

// Called when a plan is destroyed.  Only memory that is cached AND unused counts against the limit: a trim releases
// physical memory back to the driver (and the next plan pays for mapping it again, ~100 ms per GB), so it must not
// fire while plans are being created and destroyed in a steady rhythm -- only when a process that evaluated something
// big sits on more than WEALY_POOL_KEEP_MB of idle scratch.
static void pool_trim() {
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64 || !g_pools[dev]) return;
  const size_t keep = (size_t)env_int("WEALY_POOL_KEEP_MB", 4096) << 20;
  cuuint64_t reserved = 0, used = 0;
  if (cudaMemPoolGetAttribute(g_pools[dev], cudaMemPoolAttrReservedMemCurrent, &reserved) != cudaSuccess ||
      cudaMemPoolGetAttribute(g_pools[dev], cudaMemPoolAttrUsedMemCurrent, &used) != cudaSuccess) {
    cudaGetLastError();
    return;
  }
  if (reserved > used && (size_t)(reserved - used) > keep) cudaMemPoolTrimTo(g_pools[dev], (size_t)used + keep);
}

extern "C" int wealy_pool_release(void) {
  int dev = 0;
  CU_TRY(cudaGetDevice(&dev));
  {
    std::lock_guard<std::mutex> lock(g_big_mu);
    for (size_t k = 0; k < g_big.size();) {
      if (g_big[k].dev != dev) { ++k; continue; }
      cudaFreeAsync(g_big[k].ptr, g_big[k].stream);
      cudaEventDestroy(g_big[k].released);
      g_big.erase(g_big.begin() + k);
    }
  }
  CU_TRY(cudaDeviceSynchronize());  // every stream-ordered free has happened
  if (dev >= 0 && dev < 64 && g_pools[dev]) CU_TRY(cudaMemPoolTrimTo(g_pools[dev], 0));
  return WEALY_OK;
}

extern "C" int wealy_pool_stats(int64_t* reserved_bytes, int64_t* used_bytes, int64_t* reserved_high, int64_t* used_high) {
  int dev = 0;
  CU_TRY(cudaGetDevice(&dev));
  cuuint64_t v[4] = {0, 0, 0, 0};
  if (dev >= 0 && dev < 64 && g_pools[dev]) {
    CU_TRY(cudaMemPoolGetAttribute(g_pools[dev], cudaMemPoolAttrReservedMemCurrent, &v[0]));
    CU_TRY(cudaMemPoolGetAttribute(g_pools[dev], cudaMemPoolAttrUsedMemCurrent, &v[1]));
    CU_TRY(cudaMemPoolGetAttribute(g_pools[dev], cudaMemPoolAttrReservedMemHigh, &v[2]));
    CU_TRY(cudaMemPoolGetAttribute(g_pools[dev], cudaMemPoolAttrUsedMemHigh, &v[3]));
  }
  {
    // blocks parked in the library's free list are idle scratch, not memory in use
    std::lock_guard<std::mutex> lock(g_big_mu);
    for (const BigBlock& x : g_big)
      if (x.dev == dev && v[1] >= x.bytes) v[1] -= x.bytes;
  }
  if (reserved_bytes) *reserved_bytes = (int64_t)v[0];
  if (used_bytes) *used_bytes = (int64_t)v[1];
  if (reserved_high) *reserved_high = (int64_t)v[2];
  if (used_high) *used_high = (int64_t)v[3];
  return WEALY_OK;
}

// temporaries of one host function: freed (stream-ordered) on every return path
struct TempAllocs {
  cudaStream_t s;
  void* ptrs[16];
  int n = 0;
  explicit TempAllocs(cudaStream_t stream) : s(stream) {}
  cudaError_t alloc(void** ptr, size_t bytes) {
    *ptr = nullptr;
    if (n >= 16) return cudaErrorMemoryAllocation;
    cudaError_t e = dev_alloc(ptr, bytes, s);
    if (e == cudaSuccess) ptrs[n++] = *ptr;
    return e;
  }
  ~TempAllocs() {
    for (int k = 0; k < n; ++k) dev_free(ptrs[k], s);
  }
};

// ------------------------------------------------------------------------------------------
// TMA descriptors (driver entry point fetched through the runtime: no link-time libcuda dependency)
// ------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// fp16 plane [rows][d_pad] row-major; box = [box_rows][block_k] with (2 * block_k)-byte swizzle
static int make_plane_tmap(CUtensorMap* m, const void* base, int64_t rows, int64_t d_pad, int box_rows, int block_k,
                           int row_stride = 1) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return fail(WEALY_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[2] = {(cuuint64_t)d_pad, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)d_pad * 2};
  // row_stride > 1: every row_stride-th row of a (box_rows * row_stride)-row window lands in the box_rows smem rows
  cuuint32_t box[2] = {(cuuint32_t)block_k, (cuuint32_t)(box_rows * row_stride)};
  cuuint32_t estr[2] = {1, (cuuint32_t)row_stride};
  const CUtensorMapSwizzle sw = block_k == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(WEALY_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
  return WEALY_OK;
}

// ------------------------------------------------------------------------------------------
// operand planes
// ------------------------------------------------------------------------------------------
struct Planes {
  __half* hi = nullptr;
  __half* lo = nullptr;    // null in single-pass mode
  float* norm = nullptr;   // raw L2 norm per row
  float* scale = nullptr;  // epilogue row factor (power of two in RAW mode, 1 otherwise)
  float* sq = nullptr;     // squared L2 norm per row
  int64_t rows = 0;
  int64_t d_pad = 0;
};

static int64_t pad_k(int64_t d) { return ceil_div(d, 64) * 64; }

static size_t planes_bytes(int64_t rows, int64_t d, int passes) {
  const size_t plane = align_up((size_t)rows * pad_k(d) * 2, 1024);
  return plane * (passes == 3 ? 2 : 1) + 3 * align_up((size_t)rows * 4, 256);
}

// carve planes out of a workspace cursor
static void carve_planes(Planes& p, uint8_t*& cur, int64_t rows, int64_t d, int passes) {
  const size_t plane = align_up((size_t)rows * pad_k(d) * 2, 1024);
  p.rows = rows;
  p.d_pad = pad_k(d);
  p.hi = reinterpret_cast<__half*>(cur); cur += plane;
  p.lo = nullptr;
  if (passes == 3) { p.lo = reinterpret_cast<__half*>(cur); cur += plane; }
  const size_t vec = align_up((size_t)rows * 4, 256);
  p.norm = reinterpret_cast<float*>(cur); cur += vec;
  p.scale = reinterpret_cast<float*>(cur); cur += vec;
  p.sq = reinterpret_cast<float*>(cur); cur += vec;
}

static int launch_prep(const void* x, int64_t ld, int64_t n, int64_t d, int dtype, int mode, float eps,
                       const Planes& p, __half* hi_t, __half* lo_t, int64_t ld_t, ZStats* stats, int stats_on_scaled,
                       cudaStream_t s, const int* gather = nullptr, int spread_n = 0) {
  if (n == 0) return WEALY_OK;
  const int threads = 256;
  const unsigned blocks = (unsigned)ceil_div(n * 32, threads);
#define PREP_ARGS (long long)ld, (int)n, (int)d, (int)p.d_pad, mode, eps, stats_on_scaled, p.hi, p.lo, hi_t, lo_t, \
                  (long long)ld_t, p.norm, p.scale, p.sq, stats, gather, spread_n
  switch (dtype) {
    case WEALY_F32: prep_rows_kernel<float><<<blocks, threads, 0, s>>>((const float*)x, PREP_ARGS); break;
    case WEALY_F16: prep_rows_kernel<__half><<<blocks, threads, 0, s>>>((const __half*)x, PREP_ARGS); break;
    case WEALY_BF16: prep_rows_kernel<__nv_bfloat16><<<blocks, threads, 0, s>>>((const __nv_bfloat16*)x, PREP_ARGS); break;
    default: return fail(WEALY_ERR_BAD_ARG, "unknown element type %d", dtype);
  }
#undef PREP_ARGS
  CU_TRY(cudaGetLastError());
  return WEALY_OK;
}

// ------------------------------------------------------------------------------------------
// contraction launcher
// ------------------------------------------------------------------------------------------
// per-launch work counters of the dynamic unit scheduler: {next unit, CTAs through} pairs, zero at load time and reset
// by the last CTA of every launch (gemm_core.cuh: release_unit_counter) -- no memset in front of a launch.  A slot is
// reused after 2048 launches of this thread's device, long after its previous kernel has retired.
__device__ int g_unit_counters[4096];

static int next_unit_counter(int** out, cudaStream_t s) {
  (void)s;
  static thread_local int* base[64] = {nullptr};
  static int seq = 0;
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64) return fail(WEALY_ERR_UNSUPPORTED, "device index %d", dev);
  if (!base[dev]) CU_TRY(cudaGetSymbolAddress(reinterpret_cast<void**>(&base[dev]), g_unit_counters));
  const int slot = __atomic_fetch_add(&seq, 1, __ATOMIC_RELAXED) & 2047;
  *out = base[dev] + 2 * slot;
  return WEALY_OK;
}

static void fill_shape(GemmShape& sh, int64_t m, int64_t n, int64_t d_pad, int block_k, int max_chunks,
                       int tiles_per_unit = 0) {
  sh.m_rows = (int)m;
  sh.n_cols = (int)n;
  sh.k_blocks = (int)(d_pad / block_k);
  sh.n_row_blocks = (int)ceil_div(m, kTileM);
  sh.n_col_tiles = (int)ceil_div(n, kTileN);
  // enough units for ~16 rounds of the persistent grid (tail quantisation < 4 %), but never more
  // chunks than column tiles; CTAs resident together sweep the same chunk (L2 reuse of candidates)
  const int64_t target_units = (int64_t)num_sms() * env_int("WEALY_ROUNDS", 16);
  int64_t chunks = ceil_div(target_units, sh.n_row_blocks > 0 ? sh.n_row_blocks : 1);
  // short units (a few column tiles) keep the CTAs that share candidate tiles within one unit of each other
  if (tiles_per_unit > 0 && chunks < ceil_div(sh.n_col_tiles, tiles_per_unit)) chunks = ceil_div(sh.n_col_tiles, tiles_per_unit);
  if (chunks > sh.n_col_tiles) chunks = sh.n_col_tiles;
  if (chunks > max_chunks) chunks = max_chunks;
  if (chunks < 1) chunks = 1;
  sh.tiles_per_chunk = (int)ceil_div(sh.n_col_tiles, chunks);
  if (sh.tiles_per_chunk < 1) sh.tiles_per_chunk = 1;
  sh.n_col_chunks = (int)ceil_div(sh.n_col_tiles, sh.tiles_per_chunk);
  if (sh.n_col_chunks < 1) sh.n_col_chunks = 1;
  // row blocks per scheduling group: the CTAs resident together cover group_rows row blocks x all chunks
  int gr = env_int("WEALY_GROUP_ROWS", 0);
  if (gr <= 0) gr = num_sms() / (sh.n_col_chunks < 4 ? sh.n_col_chunks : 4);  // ~4 chunks in flight per group
  if (gr < 1) gr = 1;
  if (gr > sh.n_row_blocks) gr = sh.n_row_blocks > 0 ? sh.n_row_blocks : 1;
  sh.group_rows = gr;
  sh.sym = 0;
  sh.rb_stride = 1;
  sh.rb_offset = 0;
  sh.unit_counter = nullptr;
  sh.win0 = 0;
  sh.win1 = 0x7fffffff;
  sh.skip0 = sh.skip1 = 0;
}

template <class Epi, int kPasses, int kBlockK, int kEpiWarps, int kMaxStages = 8>
static int launch_gemm_t(const Planes& a, const Planes& b, const GemmShape& sh, const typename Epi::Params& ep,
                         cudaStream_t s) {
  using SM = GemmSmem<kPasses, kBlockK, kMaxStages>;
  GemmTmaps maps;
  memset(&maps, 0, sizeof(maps));
  W_TRY(make_plane_tmap(&maps.a_hi, a.hi, a.rows, a.d_pad, kTileM, kBlockK));
  W_TRY(make_plane_tmap(&maps.b_hi, b.hi, b.rows, b.d_pad, kTileN, kBlockK));
  if (kPasses == 3) {
    W_TRY(make_plane_tmap(&maps.a_lo, a.lo, a.rows, a.d_pad, kTileM, kBlockK));
    W_TRY(make_plane_tmap(&maps.b_lo, b.lo, b.rows, b.d_pad, kTileN, kBlockK));
  } else {
    maps.a_lo = maps.a_hi;
    maps.b_lo = maps.b_hi;
  }
  auto kern = gemm_kernel<Epi, kPasses, kBlockK, kEpiWarps, kMaxStages>;
  constexpr int kSmemBytes = SM::total(kEpiWarps, Epi::kWarpScratchBytes, Epi::kCtaScratchBytes);
  static_assert(kSmemBytes <= 227 * 1024, "shared memory budget");
  CU_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
  const int n_units = sh.n_row_blocks * sh.n_col_chunks;
  if (n_units == 0) return WEALY_OK;
  const int grid = n_units < num_sms() ? n_units : num_sms();
  GemmShape shl = sh;
  W_TRY(next_unit_counter(&shl.unit_counter, s));
  kern<<<grid, 64 + kEpiWarps * 32, kSmemBytes, s>>>(maps, shl, ep);
  CU_TRY(cudaGetLastError());
  return WEALY_OK;
}

// CTA-pair kernel (gemm_core2.cuh): sh.n_row_blocks / group_rows / rb_stride / rb_offset are in SUPER row blocks
template <class Epi, int kPasses, int kBlockK, int kEpiWarps = 8, bool kDyn = false>
static int launch_gemm_pair(const Planes& a, const GemmShape& sh, const typename Epi::Params& ep, cudaStream_t s,
                            const Planes* b_planes = nullptr, int max_pairs = 0) {
  constexpr int kStages = 4;
  const Planes& b = b_planes ? *b_planes : a;  // (the symmetric sweep contracts one set of planes with itself)
  const int il = (sh.sym & 2) ? 2 : 1;  // row stride of the A boxes
  using SM = PairSmem<kPasses, kBlockK, kStages>;
  GemmTmaps maps;
  memset(&maps, 0, sizeof(maps));
  // A side: the two CTAs of a pair take the even / odd rows of a 256-row super block (row-strided boxes), so that
  // neighbouring rows -- same clique, same "hotness" -- are split evenly between the two coupled epilogues
  W_TRY(make_plane_tmap(&maps.a_hi, a.hi, a.rows, a.d_pad, kTileM, kBlockK, il));
  W_TRY(make_plane_tmap(&maps.b_hi, b.hi, b.rows, b.d_pad, kTileM, kBlockK));
  if (kPasses == 3) {
    W_TRY(make_plane_tmap(&maps.a_lo, a.lo, a.rows, a.d_pad, kTileM, kBlockK, il));
    W_TRY(make_plane_tmap(&maps.b_lo, b.lo, b.rows, b.d_pad, kTileM, kBlockK));
  } else {
    maps.a_lo = maps.a_hi;
    maps.b_lo = maps.b_hi;
  }
  auto kern = gemm_pair_kernel<Epi, kPasses, kBlockK, kEpiWarps, kStages, kDyn>;
  constexpr int kSmemBytes = SM::total(kEpiWarps, Epi::kWarpScratchBytes, Epi::kCtaScratchBytes);
  static_assert(kSmemBytes <= 227 * 1024, "shared memory budget");
  CU_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
  const int n_units = sh.n_row_blocks * sh.n_col_chunks;
  if (n_units == 0) return WEALY_OK;
  int pairs = num_sms() / 2;
  if (max_pairs > 0 && max_pairs < pairs) pairs = max_pairs;  // (SMs left to another resident kernel)
  const int grid = 2 * (n_units < pairs ? n_units : pairs);
  GemmShape shl = sh;
  W_TRY(next_unit_counter(&shl.unit_counter, s));
  kern<<<grid, 64 + kEpiWarps * 32, kSmemBytes, s>>>(maps, shl, ep);
  CU_TRY(cudaGetLastError());
  return WEALY_OK;
}

// Rectangle sweeps (queries != corpus, streaming top-k, chunked tracks) on the CTA-pair core: 256 x 256 tiles per pair
// of SMs, each SM loads its 128 query rows and half of the tile's candidate rows -- 2/3 of the L2 -> shared-memory
// traffic of the single-CTA kernel, which is what bounds these sweeps (WEALY_RECT_PAIR=0 selects the single-CTA kernel).
template <class Epi>
static int launch_gemm_rect(int passes, const Planes& a, const Planes& b, GemmShape& sh, const typename Epi::Params& ep,
                            cudaStream_t s, int shard_rank = 0, int shard_world = 1);

// Multi-GPU sweeps: restrict a launch shape to the row blocks rb = shard_rank (mod shard_world) -- round-robin, so that
// the triangle of a symmetric sweep is shared evenly.  Applied to the shape the kernel reads (super row blocks on the
// CTA-pair core), after any halving.
static void shard_row_blocks(GemmShape& sh, int shard_rank, int shard_world) {
  if (shard_world <= 1) return;
  const int total_owned = sh.n_row_blocks;
  sh.rb_stride = shard_world;
  sh.rb_offset = shard_rank;
  sh.n_row_blocks = shard_rank < total_owned ? (int)ceil_div(total_owned - shard_rank, shard_world) : 0;
  if (sh.group_rows > sh.n_row_blocks) sh.group_rows = sh.n_row_blocks > 0 ? sh.n_row_blocks : 1;
}

template <class Epi>
static int launch_gemm(int passes, const Planes& a, const Planes& b, GemmShape& sh, const typename Epi::Params& ep,
                       cudaStream_t s) {
  if (passes == 3) {
    if (a.lo == nullptr || b.lo == nullptr) return fail(WEALY_ERR_BAD_ARG, "3-pass contraction needs lo planes");
    return launch_gemm_t<Epi, 3, 64, 8>(a, b, sh, ep, s);
  }
  if (passes == 1) return launch_gemm_t<Epi, 1, 64, 8>(a, b, sh, ep, s);
  return fail(WEALY_ERR_BAD_ARG, "passes must be 1 or 3, got %d", passes);
}

template <class Epi>
static int launch_gemm_rect(int passes, const Planes& a, const Planes& b, GemmShape& sh, const typename Epi::Params& ep,
                            cudaStream_t s, int shard_rank, int shard_world) {
  if (env_int("WEALY_RECT_PAIR", 1) == 0 || sh.n_row_blocks < 2) {
    GemmShape shs = sh;
    shard_row_blocks(shs, shard_rank, shard_world);
    return launch_gemm<Epi>(passes, a, b, shs, ep, s);
  }
  GemmShape shp = sh;
  shp.n_row_blocks = (sh.n_row_blocks + 1) / 2;  // super row blocks of 256 queries
  shp.group_rows = (sh.group_rows + 1) / 2;
  shard_row_blocks(shp, shard_rank, shard_world);
  if (passes == 3) {
    if (a.lo == nullptr || b.lo == nullptr) return fail(WEALY_ERR_BAD_ARG, "3-pass contraction needs lo planes");
    shp.k_blocks = (int)(a.d_pad / 32);
    return launch_gemm_pair<Epi, 3, 32, 8, false>(a, shp, ep, s, &b);
  }
  if (passes == 1) return launch_gemm_pair<Epi, 1, 64, 8, false>(a, shp, ep, s, &b);
  return fail(WEALY_ERR_BAD_ARG, "passes must be 1 or 3, got %d", passes);
}

// ------------------------------------------------------------------------------------------
// a1 / a2: materialised matrix
// ------------------------------------------------------------------------------------------
extern "C" size_t wealy_sim_matrix_workspace_bytes(int64_t n, int64_t m, int64_t d, int passes) {
  if (n < 0 || m < 0 || d <= 0) return 0;
  return planes_bytes(n, d, passes) + planes_bytes(m, d, passes) + 4096;
}

extern "C" int wealy_sim_matrix(const void* x, int64_t n, int64_t ldx, const void* y, int64_t m, int64_t ldy,
                                int64_t d, int in_dtype, int mode, float eps, float post, int passes, void* out,
                                int64_t ld_out, int out_dtype, void* workspace, size_t workspace_bytes, void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  if (n < 0 || m < 0 || d <= 0) return fail(WEALY_ERR_BAD_ARG, "bad shape n=%lld m=%lld d=%lld", (long long)n, (long long)m, (long long)d);
  if (n == 0 || m == 0) return WEALY_OK;
  if (!x || !y || !out || !workspace) return fail(WEALY_ERR_BAD_ARG, "null pointer");
  if (mode < WEALY_MODE_COSSIM || mode > WEALY_MODE_EUC) return fail(WEALY_ERR_BAD_ARG, "unknown mode %d", mode);
  if (passes != 1 && passes != 3) return fail(WEALY_ERR_BAD_ARG, "passes must be 1 or 3");
  if (n >= (1ll << 31) - 256 || m >= (1ll << 31) - 256) return fail(WEALY_ERR_UNSUPPORTED, "more than 2^31 rows");
  if (workspace_bytes < wealy_sim_matrix_workspace_bytes(n, m, d, passes))
    return fail(WEALY_ERR_WORKSPACE, "workspace too small: %zu < %zu", workspace_bytes,
                wealy_sim_matrix_workspace_bytes(n, m, d, passes));
  uint8_t* cur = reinterpret_cast<uint8_t*>(align_up((size_t)workspace, 1024));
  Planes px, py;
  carve_planes(px, cur, n, d, passes);
  const bool same = (x == y && n == m && ldx == ldy);
  if (same) py = px; else carve_planes(py, cur, m, d, passes);
  const bool cosine = (mode == WEALY_MODE_COSSIM || mode == WEALY_MODE_COS);
  const int pmode = cosine ? kPrepL2AddEps : kPrepRawPow2;
  W_TRY(launch_prep(x, ldx, n, d, in_dtype, pmode, eps, px, nullptr, nullptr, 0, nullptr, 0, s));
  if (!same) W_TRY(launch_prep(y, ldy, m, d, in_dtype, pmode, eps, py, nullptr, nullptr, 0, nullptr, 0, s));

  StoreParams sp;
  sp.out = out;
  sp.ld = ld_out;
  sp.mode = mode;
  sp.out_dtype = out_dtype;
  sp.post = post;
  sp.rscale = cosine ? nullptr : px.scale;
  sp.cscale = cosine ? nullptr : py.scale;
  sp.rsq = px.sq;
  sp.csq = py.sq;
  GemmShape sh;
  fill_shape(sh, n, m, px.d_pad, 64, 1 << 20);
  return launch_gemm<StoreEpi>(passes, px, py, sh, sp, s);
}

// float64 operands (the reference returns the input dtype): CUDA-core DGEMM with the same mode epilogue.
// workspace: 2 (n + m) doubles.
extern "C" size_t wealy_sim_matrix_f64_workspace_bytes(int64_t n, int64_t m) {
  if (n < 0 || m < 0) return 0;
  return (size_t)(2 * (n + m)) * 8 + 256;
}

extern "C" int wealy_sim_matrix_f64(const double* x, int64_t n, int64_t ldx, const double* y, int64_t m, int64_t ldy, int64_t d,
                                    int mode, double eps, double post, double* out, int64_t ld_out, void* workspace,
                                    size_t workspace_bytes, void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  if (n < 0 || m < 0 || d <= 0) return fail(WEALY_ERR_BAD_ARG, "bad shape n=%lld m=%lld d=%lld", (long long)n, (long long)m, (long long)d);
  if (n == 0 || m == 0) return WEALY_OK;
  if (!x || !y || !out || !workspace) return fail(WEALY_ERR_BAD_ARG, "null pointer");
  if (mode < WEALY_MODE_COSSIM || mode > WEALY_MODE_EUC) return fail(WEALY_ERR_BAD_ARG, "unknown mode %d", mode);
  if (n >= (1ll << 31) - 256 || m >= (1ll << 31) - 256 || m > 64ll * 65535 * 64) return fail(WEALY_ERR_UNSUPPORTED, "too many rows");
  if (workspace_bytes < wealy_sim_matrix_f64_workspace_bytes(n, m)) return fail(WEALY_ERR_WORKSPACE, "workspace too small");
  double* xn = reinterpret_cast<double*>(align_up((size_t)workspace, 16));
  double* xs = xn + n;
  double* yn = xs + n;
  double* ys = yn + m;
  row_norm_f64_kernel<<<(unsigned)ceil_div(n * 32, 256), 256, 0, s>>>(x, (long long)ldx, (int)n, (int)d, xn, xs);
  row_norm_f64_kernel<<<(unsigned)ceil_div(m * 32, 256), 256, 0, s>>>(y, (long long)ldy, (int)m, (int)d, yn, ys);
  dim3 grid((unsigned)ceil_div(m, 64), (unsigned)ceil_div(n, 64));
  if (grid.y > 65535) return fail(WEALY_ERR_UNSUPPORTED, "too many rows for the float64 path");
  sim_matrix_f64_kernel<<<grid, 256, 0, s>>>(x, (long long)ldx, (int)n, y, (long long)ldy, (int)m, (int)d, mode, eps, post, xn, xs, yn,
                                             ys, out, (long long)ld_out);
  CU_TRY(cudaGetLastError());
  return WEALY_OK;
}

// ------------------------------------------------------------------------------------------
// a1 under autograd (lib/losses.py:45 differentiates through pairwise_distance_matrix): gradient of the cosine
// modes.  S = X^ Y^T with x^ = x / (|x| + eps):  dX^ = G Y^,  dY^ = G^T X^,  then the normalisation Jacobian.
// Both products run on the contraction core: the gradient matrix (and its transpose) are split into fp16 hi/lo
// planes with an exact power-of-two row scale, the normalised operands are transposed into K-major planes.
// ------------------------------------------------------------------------------------------
static size_t tplane_bytes(int64_t rows, int64_t k, int passes) {
  return align_up((size_t)rows * pad_k(k) * 2, 1024) * (passes == 3 ? 2 : 1);
}

extern "C" size_t wealy_sim_matrix_backward_workspace_bytes(int64_t n, int64_t m, int64_t d, int passes) {
  if (n <= 0 || m <= 0 || d <= 0) return 0;
  return planes_bytes(n, d, passes) + planes_bytes(m, d, passes) + planes_bytes(n, m, passes) + planes_bytes(m, n, passes) +
         tplane_bytes(d, n, passes) + tplane_bytes(d, m, passes) + align_up((size_t)n * d * 4, 1024) +
         align_up((size_t)m * d * 4, 1024) + 8192;
}

template <typename T>
static void launch_jacobian(const void* z, int64_t ldz, int64_t rows, int64_t d, float eps, const float* norm, const float* du,
                            const float* scal, void* dz, int64_t ld_dz, cudaStream_t s) {
  loss_jacobian_kernel<T><<<(unsigned)ceil_div(rows * 32, 256), 256, 0, s>>>(kLossNtxent, eps, (const T*)z, (long long)ldz, (int)rows,
                                                                           (int)d, norm, du, scal, nullptr, (T*)dz,
                                                                           (long long)ld_dz);
}

__global__ void fill_f32_kernel(float* p, float v, int n) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) p[t] = v;
}

extern "C" int wealy_sim_matrix_backward(const void* x, int64_t n, int64_t ldx, const void* y, int64_t m, int64_t ldy,
                                         int64_t d, int in_dtype, int mode, float eps, int passes, const void* grad,
                                         int64_t ld_grad, const void* grad_t, int64_t ld_grad_t, void* dx, int64_t ld_dx,
                                         void* dy, int64_t ld_dy, void* workspace, size_t workspace_bytes, void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  if (n <= 0 || m <= 0 || d <= 0) return fail(WEALY_ERR_BAD_ARG, "bad shape n=%lld m=%lld d=%lld", (long long)n, (long long)m, (long long)d);
  if (!x || !y || !grad || !grad_t || !dx || !dy || !workspace) return fail(WEALY_ERR_BAD_ARG, "null pointer");
  if (mode != WEALY_MODE_COSSIM && mode != WEALY_MODE_COS)
    return fail(WEALY_ERR_UNSUPPORTED, "the gradient is built for the cosine modes (cos / cossim)");
  if (passes != 1 && passes != 3) return fail(WEALY_ERR_BAD_ARG, "passes must be 1 or 3");
  if (workspace_bytes < wealy_sim_matrix_backward_workspace_bytes(n, m, d, passes)) return fail(WEALY_ERR_WORKSPACE, "workspace too small");
  uint8_t* cur = reinterpret_cast<uint8_t*>(align_up((size_t)workspace, 1024));
  Planes px, py, pg, pgt;
  carve_planes(px, cur, n, d, passes);
  carve_planes(py, cur, m, d, passes);
  carve_planes(pg, cur, n, m, passes);    // G   [n][m_pad], row scale 2^e
  carve_planes(pgt, cur, m, n, passes);   // G^T [m][n_pad]
  const int64_t n_pad = pad_k(n), m_pad = pad_k(m);
  auto carve_t = [&](__half*& h, __half*& l, int64_t k) {
    const size_t plane = align_up((size_t)d * pad_k(k) * 2, 1024);
    h = reinterpret_cast<__half*>(cur); cur += plane;
    l = nullptr;
    if (passes == 3) { l = reinterpret_cast<__half*>(cur); cur += plane; }
  };
  __half *xt_hi, *xt_lo, *yt_hi, *yt_lo;
  carve_t(xt_hi, xt_lo, n);  // X^T [d][n_pad]
  carve_t(yt_hi, yt_lo, m);  // Y^T [d][m_pad]
  float* dxh = reinterpret_cast<float*>(cur); cur += align_up((size_t)n * d * 4, 1024);
  float* dyh = reinterpret_cast<float*>(cur); cur += align_up((size_t)m * d * 4, 1024);
  float* scal = reinterpret_cast<float*>(cur); cur += 256;

  W_TRY(launch_prep(x, ldx, n, d, in_dtype, kPrepL2AddEps, eps, px, nullptr, nullptr, 0, nullptr, 0, s));
  W_TRY(launch_prep(y, ldy, m, d, in_dtype, kPrepL2AddEps, eps, py, nullptr, nullptr, 0, nullptr, 0, s));
  W_TRY(launch_prep(grad, ld_grad, n, m, in_dtype, kPrepRawPow2, 0.f, pg, nullptr, nullptr, 0, nullptr, 0, s));
  W_TRY(launch_prep(grad_t, ld_grad_t, m, n, in_dtype, kPrepRawPow2, 0.f, pgt, nullptr, nullptr, 0, nullptr, 0, s));
  {
    dim3 gx((unsigned)ceil_div(n_pad, 32), (unsigned)ceil_div(d, 32), px.lo ? 2 : 1);
    transpose_plane_kernel<<<gx, 256, 0, s>>>(px.hi, px.lo, (int)n, (int)d, (long long)px.d_pad, xt_hi, xt_lo, (long long)n_pad);
    dim3 gy((unsigned)ceil_div(m_pad, 32), (unsigned)ceil_div(d, 32), py.lo ? 2 : 1);
    transpose_plane_kernel<<<gy, 256, 0, s>>>(py.hi, py.lo, (int)m, (int)d, (long long)py.d_pad, yt_hi, yt_lo, (long long)m_pad);
    fill_f32_kernel<<<1, 32, 0, s>>>(scal, mode == WEALY_MODE_COS ? -1.f : 1.f, 1);  // d(1 - S) = -dS
    CU_TRY(cudaGetLastError());
  }
  auto product = [&](const Planes& g, __half* bt_hi, __half* bt_lo, int64_t rows, int64_t k_pad, float* out) -> int {
    Planes pa = g, pb;
    pa.rows = rows;
    pb.hi = bt_hi; pb.lo = bt_lo; pb.rows = d; pb.d_pad = k_pad;
    StoreParams sp;
    memset(&sp, 0, sizeof(sp));
    sp.out = out;
    sp.ld = d;
    sp.mode = kSimDotsim;   // s * row scale (the transposed operands carry no scale)
    sp.out_dtype = kOutF32;
    sp.post = 1.f;
    sp.rscale = g.scale;
    GemmShape sh;
    fill_shape(sh, rows, d, k_pad, 64, 1 << 20);
    return launch_gemm<StoreEpi>(passes, pa, pb, sh, sp, s);
  };
  W_TRY(product(pg, yt_hi, yt_lo, n, m_pad, dxh));   // dX^ = G Y^
  W_TRY(product(pgt, xt_hi, xt_lo, m, n_pad, dyh));  // dY^ = G^T X^
  switch (in_dtype) {
    case WEALY_F32:
      launch_jacobian<float>(x, ldx, n, d, eps, px.norm, dxh, scal, dx, ld_dx, s);
      launch_jacobian<float>(y, ldy, m, d, eps, py.norm, dyh, scal, dy, ld_dy, s);
      break;
    case WEALY_F16:
      launch_jacobian<__half>(x, ldx, n, d, eps, px.norm, dxh, scal, dx, ld_dx, s);
      launch_jacobian<__half>(y, ldy, m, d, eps, py.norm, dyh, scal, dy, ld_dy, s);
      break;
    case WEALY_BF16:
      launch_jacobian<__nv_bfloat16>(x, ldx, n, d, eps, px.norm, dxh, scal, dx, ld_dx, s);
      launch_jacobian<__nv_bfloat16>(y, ldy, m, d, eps, py.norm, dyh, scal, dy, ld_dy, s);
      break;
    default: return fail(WEALY_ERR_BAD_ARG, "unknown element type %d", in_dtype);
  }
  CU_TRY(cudaGetLastError());
  return WEALY_OK;
}

// Gradient of the dot modes (no normalisation): dX = G Y, dY = G^T X.  The caller passes the gradient and its
// transpose (already negated for mode "dot" = 1 - x.y) and the TRANSPOSED operands xt [d][n], yt [d][m]: every
// matrix is split row-wise with an exact power-of-two scale, so the products are plain K-major contractions.
extern "C" size_t wealy_dot_matrix_backward_workspace_bytes(int64_t n, int64_t m, int64_t d, int passes) {
  if (n <= 0 || m <= 0 || d <= 0) return 0;
  return planes_bytes(n, m, passes) + planes_bytes(m, n, passes) + planes_bytes(d, n, passes) + planes_bytes(d, m, passes) + 8192;
}

extern "C" int wealy_dot_matrix_backward(const void* grad, int64_t ld_grad, const void* grad_t, int64_t ld_grad_t,
                                         const void* xt, int64_t ld_xt, const void* yt, int64_t ld_yt, int64_t n, int64_t m,
                                         int64_t d, int dtype, int passes, void* dx, int64_t ld_dx, void* dy, int64_t ld_dy,
                                         void* workspace, size_t workspace_bytes, void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  if (n <= 0 || m <= 0 || d <= 0) return fail(WEALY_ERR_BAD_ARG, "bad shape n=%lld m=%lld d=%lld", (long long)n, (long long)m, (long long)d);
  if (!grad || !grad_t || !xt || !yt || !dx || !dy || !workspace) return fail(WEALY_ERR_BAD_ARG, "null pointer");
  if (passes != 1 && passes != 3) return fail(WEALY_ERR_BAD_ARG, "passes must be 1 or 3");
  if (workspace_bytes < wealy_dot_matrix_backward_workspace_bytes(n, m, d, passes)) return fail(WEALY_ERR_WORKSPACE, "workspace too small");
  uint8_t* cur = reinterpret_cast<uint8_t*>(align_up((size_t)workspace, 1024));
  Planes pg, pgt, pxt, pyt;
  carve_planes(pg, cur, n, m, passes);    // G    [n][m_pad]
  carve_planes(pgt, cur, m, n, passes);   // G^T  [m][n_pad]
  carve_planes(pxt, cur, d, n, passes);   // X^T  [d][n_pad]
  carve_planes(pyt, cur, d, m, passes);   // Y^T  [d][m_pad]
  W_TRY(launch_prep(grad, ld_grad, n, m, dtype, kPrepRawPow2, 0.f, pg, nullptr, nullptr, 0, nullptr, 0, s));
  W_TRY(launch_prep(grad_t, ld_grad_t, m, n, dtype, kPrepRawPow2, 0.f, pgt, nullptr, nullptr, 0, nullptr, 0, s));
  W_TRY(launch_prep(xt, ld_xt, d, n, dtype, kPrepRawPow2, 0.f, pxt, nullptr, nullptr, 0, nullptr, 0, s));
  W_TRY(launch_prep(yt, ld_yt, d, m, dtype, kPrepRawPow2, 0.f, pyt, nullptr, nullptr, 0, nullptr, 0, s));
  auto product = [&](const Planes& a, const Planes& b, int64_t rows, void* out, int64_t ld_out) -> int {
    StoreParams sp;
    memset(&sp, 0, sizeof(sp));
    sp.out = out;
    sp.ld = ld_out;
    sp.mode = kSimDotsim;  // s * row scale * column scale
    sp.out_dtype = dtype == WEALY_F32 ? kOutF32 : (dtype == WEALY_F16 ? kOutF16 : kOutBF16);
    sp.post = 1.f;
    sp.rscale = a.scale;
    sp.cscale = b.scale;
    GemmShape sh;
    fill_shape(sh, rows, d, a.d_pad, 64, 1 << 20);
    return launch_gemm<StoreEpi>(passes, a, b, sh, sp, s);
  };
  W_TRY(product(pg, pyt, n, dx, ld_dx));    // dX = G Y      (K = m)
  W_TRY(product(pgt, pxt, m, dy, ld_dy));   // dY = G^T X    (K = n)
  return WEALY_OK;
}

// ------------------------------------------------------------------------------------------
// a7: evaluation plan + run
// ------------------------------------------------------------------------------------------
struct wealy_eval_plan {
  int64_t nq = 0, nc = 0;
  cudaStream_t stream = nullptr;  // stream the plan was built on
  cudaStream_t last_stream = nullptr;  // stream of the last run (frees are ordered on it)
  bool same_ids = false;
  int *q_c = nullptr, *q_i = nullptr, *c_c = nullptr, *c_i = nullptr;
  int *sorted_c = nullptr, *sorted_idx = nullptr;
  int *seg_lo = nullptr, *seg_len = nullptr, *npos = nullptr;
  long long* off = nullptr;  // [nq + 1]
  int64_t total_pairs = 0, no_relevant = 0, max_relevant = 0;
  int64_t max_clique = 0;  // longest run of one clique id among the candidates
  // scratch that depends on ids only
  float *raw = nullptr, *thr = nullptr, *lim = nullptr;
  int* cnt = nullptr;
  unsigned int* hist = nullptr;
  // embedding-dependent scratch, (re)allocated when the shape grows
  void* planes_buf = nullptr;
  size_t planes_cap = 0;
  void* topk_buf = nullptr;
  size_t topk_cap = 0;
  void* tks_buf = nullptr;   // top-k in the symmetric sweep: sample operand, pre-pass lists, bounds, candidate lists
  size_t tks_cap = 0;
  int last_topk_path = 0;    // 0 none, 1 symmetric sweep, 2 rectangle sweep, 3 symmetric failed -> rectangle
  // clique-sorted view of an all-vs-all plan (same ids on both sides): the symmetric sweep runs in this row order
  // (perm = sorted_idx: sorted position -> caller's row; clique ids = sorted_c)
  int *s_i = nullptr, *s_seg_lo = nullptr, *s_seg_len = nullptr, *s_npos = nullptr;
  long long* s_off = nullptr;
  float4* s_lvl = nullptr;
  void* lvl_thr_buf = nullptr;  // all-vs-all plans: [s_lvl | thr] in one allocation (one all-reduce sums both over the ranks)
  uint2* s_cinfo = nullptr;
  unsigned char* s_dirty = nullptr;
  int64_t s_padded = 0;
  // CUDA events bracketing the fused sweep of the last run (roofline accounting in bench.py)
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  // ... and the stages around it: [0] before prep, [1] before K_pos, [2] after ap_reduce, [3] after the top-k finalize
  cudaEvent_t evs[4] = {nullptr, nullptr, nullptr, nullptr};
  bool timed = false;
  bool finished = false;  // the last run recorded the events after ap_reduce and the top-k finalize (evs[2], evs[3])
  bool last_sym = false;  // the last sweep ran in the clique-sorted view (its counters are in that CSR order)
  int staged_chunks = 0;  // chunks of the last staged prepare (0 none); > 1: the summed buffer is thr alone
  // wealy_eval_run_host: [0] "planes allocated" on the run's stream, [1 + k] "rows of part k have arrived" on the upload stream
  cudaEvent_t host_ev[1 + 8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  // wealy_eval_plan_create_host: plane rows [early_lo, end) of this matrix are already in flight on the upload stream
  // (issued while the rest of the plan was being built); -1 = none / consumed by the run
  int64_t early_lo = -1, early_ld = 0, early_d = 0;
  const void* early_z = nullptr;
  int early_dtype = 0, early_passes = 0;
  float early_eps = 0.f;
};

static cudaStream_t upload_stream();

extern "C" void wealy_eval_plan_destroy(wealy_eval_plan* p) {
  if (!p) return;
  if (p->early_lo >= 0) {  // (a plan created with an early upload and never run: the upload still writes the planes)
    cudaStream_t up = upload_stream();
    if (up) cudaStreamSynchronize(up);
  }
  void* ptrs[] = {p->q_c, p->q_i, p->sorted_c, p->sorted_idx, p->seg_lo, p->seg_len, p->npos, p->off,
                  p->raw, p->lvl_thr_buf ? nullptr : (void*)p->thr, p->lim, p->cnt, p->hist,
                  p->s_i, p->s_seg_lo, p->s_seg_len, p->s_npos, p->s_off, p->lvl_thr_buf ? p->lvl_thr_buf : (void*)p->s_lvl,
                  p->s_cinfo, p->s_dirty};
  // frees are ordered behind the last work that touched the buffers: the stream of the last run
  cudaStream_t fs = p->timed ? p->last_stream : p->stream;
  for (void* q : ptrs) dev_free(q, fs);
  big_free(p->planes_buf, p->planes_cap, fs);
  big_free(p->topk_buf, p->topk_cap, fs);
  big_free(p->tks_buf, p->tks_cap, fs);
  if (!p->same_ids) {
    dev_free(p->c_c, fs);
    dev_free(p->c_i, fs);
  }
  pool_trim();
  if (p->ev0) cudaEventDestroy(p->ev0);
  if (p->ev1) cudaEventDestroy(p->ev1);
  for (cudaEvent_t e : p->evs)
    if (e) cudaEventDestroy(e);
  for (cudaEvent_t e : p->host_ev)
    if (e) cudaEventDestroy(e);
  delete p;
}

// CSR offsets are 64-bit: the scan must ACCUMULATE in 64 bits too (one clique of ~46k versions already holds 2^31
// relevant pairs), so the int32 counts are widened on the fly.
struct WidenI32 {
  __host__ __device__ __forceinline__ long long operator()(const int& v) const { return (long long)v; }
};
using WideCounts = cub::TransformInputIterator<long long, WidenI32, const int*>;

static int plan_build(wealy_eval_plan* p, const int64_t* queries_c, const int64_t* queries_i,
                      const int64_t* candidates_c, const int64_t* candidates_i, cudaStream_t s,
                      const std::function<int()>& after_sort = nullptr) {
  const int nq = (int)p->nq, nc = (int)p->nc;
  const int T = 256;
  TempAllocs tmps(s);
  int* bad = nullptr;
  unsigned long long* totals = nullptr;
  CU_TRY(tmps.alloc((void**)&bad, 256));
  totals = reinterpret_cast<unsigned long long*>(bad + 16);
  CU_TRY(cudaMemsetAsync(bad, 0, 256, s));
  CU_TRY(dev_alloc((void**)&p->q_c, (size_t)nq * 4 + 4, s));
  CU_TRY(dev_alloc((void**)&p->q_i, (size_t)nq * 4 + 4, s));
  ids_to_i32_kernel<<<(unsigned)ceil_div(nq, T), T, 0, s>>>((const long long*)queries_c, p->q_c, nq, bad);
  ids_to_i32_kernel<<<(unsigned)ceil_div(nq, T), T, 0, s>>>((const long long*)queries_i, p->q_i, nq, bad);
  p->same_ids = (queries_c == candidates_c && queries_i == candidates_i && p->nq == p->nc);
  if (!p->same_ids && p->nq == p->nc) {
    // equal ids in distinct buffers are still an all-vs-all problem (one extra 4-byte read-back decides it)
    ids_differ_kernel<<<(unsigned)ceil_div(nq, T), T, 0, s>>>((const long long*)queries_c, (const long long*)queries_i,
                                                             (const long long*)candidates_c, (const long long*)candidates_i, nq, bad + 8);
    int differ = 1;
    CU_TRY(cudaMemcpyAsync(&differ, bad + 8, sizeof(int), cudaMemcpyDeviceToHost, s));
    CU_TRY(cudaStreamSynchronize(s));
    p->same_ids = differ == 0;
  }
  if (p->same_ids) {
    p->c_c = p->q_c;
    p->c_i = p->q_i;
  } else {
    CU_TRY(dev_alloc((void**)&p->c_c, (size_t)nc * 4 + 4, s));
    CU_TRY(dev_alloc((void**)&p->c_i, (size_t)nc * 4 + 4, s));
    ids_to_i32_kernel<<<(unsigned)ceil_div(nc, T), T, 0, s>>>((const long long*)candidates_c, p->c_c, nc, bad);
    ids_to_i32_kernel<<<(unsigned)ceil_div(nc, T), T, 0, s>>>((const long long*)candidates_i, p->c_i, nc, bad);
  }
  CU_TRY(cudaGetLastError());

  // candidates sorted by clique id (CUB radix sort: id-only preprocessing, not on the per-eval path)
  int* iota = nullptr;
  CU_TRY(tmps.alloc((void**)&iota, (size_t)nc * 4 + 4));
  CU_TRY(dev_alloc((void**)&p->sorted_c, (size_t)nc * 4 + 4, s));
  CU_TRY(dev_alloc((void**)&p->sorted_idx, (size_t)nc * 4 + 4, s));
  iota_kernel<<<(unsigned)ceil_div(nc, T), T, 0, s>>>(iota, nc);
  size_t tmp_bytes = 0;
  CU_TRY(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, p->c_c, p->sorted_c, iota, p->sorted_idx, nc, 0, 32, s));
  void* tmp = nullptr;
  CU_TRY(tmps.alloc((void**)&tmp, tmp_bytes + 16));
  CU_TRY(cub::DeviceRadixSort::SortPairs(tmp, tmp_bytes, p->c_c, p->sorted_c, iota, p->sorted_idx, nc, 0, 32, s));
  // (wealy_eval_plan_create_host: the sorted order is all the upload of the first rows needs -- it starts here, under
  // the rest of the plan)
  if (after_sort && p->same_ids) W_TRY(after_sort());

  CU_TRY(dev_alloc((void**)&p->seg_lo, (size_t)nq * 4 + 4, s));
  CU_TRY(dev_alloc((void**)&p->seg_len, (size_t)nq * 4 + 4, s));
  CU_TRY(dev_alloc((void**)&p->npos, (size_t)nq * 4 + 4, s));
  CU_TRY(dev_alloc((void**)&p->off, ((size_t)nq + 1) * 8, s));
  segment_lookup_kernel<<<(unsigned)ceil_div(nq, T), T, 0, s>>>(p->q_c, p->q_i, nq, p->sorted_c, p->sorted_idx, p->c_i,
                                                               nc, p->seg_lo, p->seg_len, p->npos, totals);
  CU_TRY(cudaGetLastError());
  // CSR offsets over the per-query number of relevant candidates
  size_t scan_bytes = 0;
  CU_TRY(cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, WideCounts(p->npos, WidenI32()), p->off, nq + 1, s));
  void* tmp2 = nullptr;
  CU_TRY(tmps.alloc((void**)&tmp2, scan_bytes + 16));
  // npos has nq valid entries; entry nq is read by the scan of nq+1 items -> zero it first
  CU_TRY(cudaMemsetAsync(p->npos + nq, 0, 4, s));
  CU_TRY(cub::DeviceScan::ExclusiveSum(tmp2, scan_bytes, WideCounts(p->npos, WidenI32()), p->off, nq + 1, s));

  // ---- clique-sorted view for the symmetric all-vs-all sweep
  void* tmp3 = nullptr;
  int *vkeys = nullptr, *vpos = nullptr, *everything = nullptr;
  if (p->same_ids) {
    const int n = nq;
    const int nrb = (int)ceil_div(n, kTileM), nct = (int)ceil_div(n, kTileN);
    p->s_padded = (int64_t)nct * kTileN + kTileN;
    CU_TRY(dev_alloc((void**)&p->s_i, (size_t)n * 4 + 4, s));
    CU_TRY(dev_alloc((void**)&p->s_seg_lo, (size_t)n * 4 + 4, s));
    CU_TRY(dev_alloc((void**)&p->s_seg_len, (size_t)n * 4 + 4, s));
    CU_TRY(dev_alloc((void**)&p->s_npos, (size_t)n * 4 + 4, s));
    CU_TRY(dev_alloc((void**)&p->s_off, ((size_t)n + 1) * 8, s));
    // (allocated below, next to the thresholds, once their number is known)
    CU_TRY(dev_alloc((void**)&p->s_cinfo, (size_t)p->s_padded * 8, s));
    CU_TRY(dev_alloc((void**)&p->s_dirty, (size_t)nrb * nct, s));
    gather_i32_kernel<<<(unsigned)ceil_div(n, T), T, 0, s>>>(p->q_i, p->sorted_idx, n, p->s_i);
    // in sorted space the clique-sorted order is the identity (iota)
    segment_lookup_kernel<<<(unsigned)ceil_div(n, T), T, 0, s>>>(p->sorted_c, p->s_i, n, p->sorted_c, iota, p->s_i, n,
                                                                p->s_seg_lo, p->s_seg_len, p->s_npos, totals + 2);
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaMemsetAsync(p->s_npos + n, 0, 4, s));
    CU_TRY(cub::DeviceScan::ExclusiveSum(tmp2, scan_bytes, WideCounts(p->s_npos, WidenI32()), p->s_off, n + 1, s));
    // tiles that need id tests: clique ranges that intersect, ragged edges, version-id collisions
    CU_TRY(cudaMemsetAsync(p->s_dirty, 0, (size_t)nrb * nct, s));
    dirty_clique_kernel<<<(unsigned)ceil_div((int64_t)nrb * nct, T), T, 0, s>>>(p->sorted_c, n, nrb, nct, p->s_dirty);
    CU_TRY(tmps.alloc((void**)&vkeys, (size_t)n * 4 + 4));
    CU_TRY(tmps.alloc((void**)&vpos, (size_t)n * 4 + 4));
    CU_TRY(tmps.alloc((void**)&everything, 16));
    CU_TRY(cudaMemsetAsync(everything, 0, 16, s));
    size_t tb = 0;
    CU_TRY(cub::DeviceRadixSort::SortPairs(nullptr, tb, p->s_i, vkeys, iota, vpos, n, 0, 32, s));
    CU_TRY(tmps.alloc(&tmp3, tb + 16));
    CU_TRY(cub::DeviceRadixSort::SortPairs(tmp3, tb, p->s_i, vkeys, iota, vpos, n, 0, 32, s));
    dirty_collision_kernel<<<(unsigned)ceil_div(n, T), T, 0, s>>>(vkeys, vpos, n, nrb, nct, p->s_dirty, everything);
    dirty_everything_kernel<<<(unsigned)ceil_div((int64_t)nrb * nct, T), T, 0, s>>>(everything, (long long)nrb * nct, p->s_dirty);
    CU_TRY(cudaGetLastError());
  }

  int bad_h[16];
  unsigned long long totals_h[5];
  long long total = 0;
  CU_TRY(cudaMemcpyAsync(bad_h, bad, sizeof(int), cudaMemcpyDeviceToHost, s));
  CU_TRY(cudaMemcpyAsync(totals_h, totals, sizeof(totals_h), cudaMemcpyDeviceToHost, s));
  CU_TRY(cudaMemcpyAsync(&total, p->off + nq, 8, cudaMemcpyDeviceToHost, s));
  CU_TRY(cudaStreamSynchronize(s));
  if (bad_h[0] != 0) return fail(WEALY_ERR_ID_RANGE, "%d clique/version ids do not fit in 32 bits", bad_h[0]);
  p->total_pairs = total;
  p->no_relevant = (int64_t)totals_h[0];
  p->max_relevant = (int64_t)totals_h[1];
  p->max_clique = (int64_t)totals_h[4];
  const size_t pairs = (size_t)(total > 0 ? total : 1);
  CU_TRY(dev_alloc((void**)&p->raw, pairs * 4, s));
  if (p->same_ids) {
    CU_TRY(dev_alloc(&p->lvl_thr_buf, (size_t)p->s_padded * 16 + pairs * 4, s));
    p->s_lvl = reinterpret_cast<float4*>(p->lvl_thr_buf);
    p->thr = reinterpret_cast<float*>(p->s_lvl + p->s_padded);
  } else {
    CU_TRY(dev_alloc((void**)&p->thr, pairs * 4, s));
  }
  CU_TRY(dev_alloc((void**)&p->hist, pairs * 4, s));
  CU_TRY(dev_alloc((void**)&p->lim, (size_t)nq * 4 + 4, s));
  CU_TRY(dev_alloc((void**)&p->cnt, (size_t)nq * 4 + 4, s));
  return WEALY_OK;
}

extern "C" int wealy_eval_plan_create(const int64_t* queries_c, const int64_t* queries_i, int64_t nq,
                                      const int64_t* candidates_c, const int64_t* candidates_i, int64_t nc,
                                      void* stream, wealy_eval_plan** plan) {
  if (!plan) return fail(WEALY_ERR_BAD_ARG, "plan output pointer is null");
  *plan = nullptr;
  if (nq <= 0 || nc <= 0) return fail(WEALY_ERR_BAD_ARG, "empty query or candidate set (nq=%lld nc=%lld)", (long long)nq, (long long)nc);
  if (!queries_c || !queries_i || !candidates_c || !candidates_i) return fail(WEALY_ERR_BAD_ARG, "null id pointer");
  if (nq >= (1ll << 31) - 256 || nc >= (1ll << 31) - 256) return fail(WEALY_ERR_UNSUPPORTED, "more than 2^31 rows");
  wealy_eval_plan* p = new wealy_eval_plan();
  p->nq = nq;
  p->nc = nc;
  p->stream = (cudaStream_t)stream;
  int st = plan_build(p, queries_c, queries_i, candidates_c, candidates_i, (cudaStream_t)stream);
  if (st != WEALY_OK) {
    wealy_eval_plan_destroy(p);
    return st;
  }
  *plan = p;
  return WEALY_OK;
}

extern "C" int wealy_eval_plan_info(const wealy_eval_plan* p, int64_t* total_pairs, int64_t* queries_without_relevant,
                                    int64_t* max_relevant) {
  if (!p) return fail(WEALY_ERR_BAD_ARG, "null plan");
  if (total_pairs) *total_pairs = p->total_pairs;
  if (queries_without_relevant) *queries_without_relevant = p->no_relevant;
  if (max_relevant) *max_relevant = p->max_relevant;
  return WEALY_OK;
}

extern "C" int wealy_eval_plan_last_sweep_ms(const wealy_eval_plan* p, float* ms) {
  if (!p || !ms) return fail(WEALY_ERR_BAD_ARG, "null pointer");
  if (!p->timed) return fail(WEALY_ERR_BAD_ARG, "the plan has not been run yet");
  CU_TRY(cudaEventSynchronize(p->ev1));
  CU_TRY(cudaEventElapsedTime(ms, p->ev0, p->ev1));
  return WEALY_OK;
}

// Candidate-list capacity per (row, part).  A row may gain up to 4 deferred chunks x 32 candidates between two
// compaction checks (k + 128 <= cap is required); the slack beyond that sets how often a list is compacted.
static int topk_capacity(int k) {
  size_t cap = align_up((size_t)(2 * k > k + 192 ? 2 * k : k + 192), 32);
  if (cap > 1024) cap = 1024;
  return (int)cap;
}

// shard_world > 1: symmetric sweep restricted to the row blocks rb = shard_rank (mod shard_world); the rank
// counts are left in the plan's histogram for the caller to sum over ranks (finish == false).
// chunks > 1 (row f1): every track has `chunks` embeddings (rows t * chunks .. of the matrices), the kS x kS chunk
// similarities are reduced to one per track pair inside the epilogue (redux: WEALY_REDUX_*), all ids / outputs per track.
// A sharded chunked sweep (shard_world > 1) takes the row blocks rb = shard_rank (mod shard_world) of the launched shape:
// the half sweep's pairs score their row and their column query, the rectangle's rows are complete -- either way the
// counters summed over the ranks are those of the whole sweep.
template <int kS>
static int launch_eval_tracks(int passes, const Planes& a, const Planes& b, GemmShape& sh, const EvalParams& ep, cudaStream_t s,
                              bool sym, int shard_rank, int shard_world) {
  if (!sym) return launch_gemm_rect<EvalTracksEpi<kS>>(passes, a, b, sh, ep, s, shard_rank, shard_world);
  // chunked all-vs-all: only the tiles that reach above the diagonal, on the CTA-pair core (super row block S = rows
  // [256 S, 256 S + 256) needs column tiles >= S); every track pair scores both its row and its column query
  GemmShape shp = sh;
  shp.n_row_blocks = (sh.n_row_blocks + 1) / 2;
  shp.group_rows = (sh.group_rows + 1) / 2;
  shp.sym = 1;
  shard_row_blocks(shp, shard_rank, shard_world);
  if (passes == 3) {
    shp.k_blocks = (int)(a.d_pad / 32);
    return launch_gemm_pair<EvalTracksSymEpi<kS>, 3, 32, 8, false>(a, shp, ep, s);
  }
  return launch_gemm_pair<EvalTracksSymEpi<kS>, 1, 64, 8, false>(a, shp, ep, s);
}

static int eval_run_impl(wealy_eval_plan* p, const void* queries_z, int64_t ld_q, const void* candidates_z,
                         int64_t ld_c, int64_t d, int dtype, float eps, int passes, int topk, float* aps,
                         float* r1s, double* sums, int64_t* topk_idx, float* topk_sim, int shard_rank,
                         int shard_world, bool finish, void* stream, int chunks = 1, int redux = WEALY_REDUX_MIN,
                         const int* q_len = nullptr, const int* c_len = nullptr, bool allow_sym_topk = true, int stage = 0,
                         int* local_idx = nullptr, int* local_cnt = nullptr) {
  // stage (sharded all-vs-all sweeps only): 0 = everything in one call; 1 = prep + the relevant similarities of THIS
  // rank's share of the queries, then return (the caller sums the threshold buffer over the ranks); 2 = the sweep,
  // on the planes and thresholds stage 1 left in the plan
  // local_cnt != NULL (wealy_eval_sweep_shard_topk): the symmetric top-k sweep over this rank's row blocks, its lists
  // finalized locally into topk_sim / local_idx / local_cnt; the rank counters stay in the plan (finish == false)
  const bool local = local_cnt != nullptr;
  cudaStream_t s = (cudaStream_t)stream;
  if (!p) return fail(WEALY_ERR_BAD_ARG, "null plan");
  if (p->early_lo >= 0) {
    // a plan created by wealy_eval_plan_create_host that is run on device embeddings after all: its early upload may
    // still be writing the planes this run is about to fill -- order the run behind it
    cudaStream_t up = upload_stream();
    if (up && p->host_ev[1]) {
      CU_TRY(cudaEventRecord(p->host_ev[1], up));
      CU_TRY(cudaStreamWaitEvent(s, p->host_ev[1], 0));
    }
    p->early_lo = -1;
  }
  if (stage != 2 && (!queries_z || !candidates_z)) return fail(WEALY_ERR_BAD_ARG, "null pointer");
  if (stage == 2) {
    if (!p->planes_buf || !p->lvl_thr_buf) return fail(WEALY_ERR_BAD_ARG, "wealy_eval_shard_sweep needs wealy_eval_shard_prepare first");
    if (chunks > 1 ? p->staged_chunks != chunks : p->staged_chunks > 1)
      return fail(WEALY_ERR_BAD_ARG, "the staged sweep needs a prepare of the same layout (%d chunks per track)", chunks);
    queries_z = candidates_z = p;  // (not dereferenced: the planes are in the plan)
  }
  if (finish && (!aps || !r1s || !sums)) return fail(WEALY_ERR_BAD_ARG, "null pointer");
  if (shard_world < 1 || shard_rank < 0 || shard_rank >= shard_world) return fail(WEALY_ERR_BAD_ARG, "bad shard %d/%d", shard_rank, shard_world);
  if (d <= 0) return fail(WEALY_ERR_BAD_ARG, "bad embedding size %lld", (long long)d);
  if (passes != 1 && passes != 3) return fail(WEALY_ERR_BAD_ARG, "passes must be 1 or 3");
  if (topk < 0 || topk > 800) return fail(WEALY_ERR_UNSUPPORTED, "topk must be in [0, 800], got %d", topk);
  if (topk > 0 && (!(local ? (void*)local_idx : (void*)topk_idx) || !topk_sim)) return fail(WEALY_ERR_BAD_ARG, "topk outputs are null");
  const int64_t nq = p->nq, nc = p->nc;
  const bool same = (queries_z == candidates_z && nq == nc && ld_q == ld_c);
  if (chunks != 1 && chunks != 2 && chunks != 4 && chunks != 8 && chunks != 16)
    return fail(WEALY_ERR_UNSUPPORTED, "chunks per track must be 1, 2, 4, 8 or 16, got %d", chunks);
  if (redux < WEALY_REDUX_MIN || redux > WEALY_REDUX_MINMEAN) return fail(WEALY_ERR_BAD_ARG, "unknown redux %d", redux);
  if ((q_len == nullptr) != (c_len == nullptr)) return fail(WEALY_ERR_BAD_ARG, "q_len and c_len go together");
  if (q_len && chunks == 1) return fail(WEALY_ERR_BAD_ARG, "chunk counts need chunks > 1");
  if ((nq * chunks) >= (1ll << 31) - 256 || (nc * chunks) >= (1ll << 31) - 256) return fail(WEALY_ERR_UNSUPPORTED, "more than 2^31 rows");
  // similarity space: distance min <-> similarity max; {inner over the candidate's chunks, outer over the query's}
  int red_inner = kRedMax, red_outer = kRedMax;
  float red_scale = 1.f;
  switch (redux) {
    case WEALY_REDUX_MIN: break;
    case WEALY_REDUX_MAX: red_inner = red_outer = kRedMin; break;
    case WEALY_REDUX_MEAN: red_inner = red_outer = kRedSum; red_scale = 1.f / (float)(chunks * chunks); break;
    case WEALY_REDUX_MEANMIN: red_inner = kRedMax; red_outer = kRedSum; red_scale = 1.f / (float)chunks; break;
    case WEALY_REDUX_MINMEAN: red_inner = kRedSum; red_outer = kRedMax; red_scale = 1.f / (float)chunks; break;
  }

  // Symmetric all-vs-all: queries ARE the candidates (same ids, same embeddings), no top-k.  Only the tiles
  // that reach above the diagonal are contracted (half the tensor work); every element scores both its row
  // query and its column query.  Runs in the plan's clique-sorted row order (eval_sym_epilogue.cuh).
  const bool can_sym = same && p->same_ids && chunks == 1 && p->total_pairs < (1ll << 31) - 8;
  // ... with top-k (topk_sym_kernels.cuh): a sampled pre-pass bounds every query's k-th best similarity from below, the
  // sweep appends what lies above the bound to per-query lists in both directions.  Worth it (and statistically sound)
  // for large sets and moderate k; everything else keeps the rectangle sweep with its streaming top-k.
  const bool sym_topk = can_sym && topk > 0 && topk <= 128 && nq >= env_int("WEALY_SYM_TOPK_MIN_ROWS", 16384) &&
                        nq >= 192ll * topk && (local || (finish && shard_world == 1)) &&
                        allow_sym_topk && env_int("WEALY_SYM_TOPK", 1) != 0;
  const bool sym = can_sym && (topk == 0 ? (shard_world > 1 || env_int("WEALY_SYM", 1) != 0) : sym_topk);
  // chunked tracks, all-vs-all: the same halving for reductions that give d(q, c) == d(c, q) (min / max / mean)
  const bool all_tracks = same && p->same_ids && chunks > 1 && topk == 0;
  const bool sym_tracks = all_tracks && red_inner == red_outer && nq * chunks > 2 * kTileM && env_int("WEALY_SYM_TRACKS", 1) != 0;
  if (local && !sym_topk)
    return fail(WEALY_ERR_UNSUPPORTED, "the sharded top-k sweep needs queries == candidates (ids and embeddings), plain "
                "embeddings, k <= 128 and N >= max(WEALY_SYM_TOPK_MIN_ROWS, 192 k), got N = %lld, k = %d", (long long)nq, topk);
  if (shard_world > 1 && !sym && !all_tracks)
    return fail(WEALY_ERR_BAD_ARG, "a sharded sweep needs queries == candidates (ids and embeddings) and no top-k");

  // operand planes (cached allocation)
  const int64_t rq = nq * chunks, rc = nc * chunks;  // embedding rows
  // the symmetric sweep stores its planes in spread order over whole 128-row blocks (gemm_core.cuh)
  const int64_t rows_q = sym ? ceil_div(nq, kTileM) * kTileM : rq;
  const size_t need = planes_bytes(rows_q, d, passes) + (same ? 0 : planes_bytes(rc, d, passes)) + 2048;
  if (need > p->planes_cap) {
    big_free(p->planes_buf, p->planes_cap, s);
    p->planes_buf = nullptr;
    p->planes_cap = 0;
    CU_TRY(big_alloc((void**)&p->planes_buf, &p->planes_cap, need, s));
  }
  uint8_t* cur = reinterpret_cast<uint8_t*>(align_up((size_t)p->planes_buf, 1024));
  Planes pq, pc;
  carve_planes(pq, cur, rows_q, d, passes);
  if (same) pc = pq; else carve_planes(pc, cur, rc, d, passes);
  if (!p->ev0) {
    CU_TRY(cudaEventCreate(&p->ev0));
    CU_TRY(cudaEventCreate(&p->ev1));
    for (cudaEvent_t& e : p->evs) CU_TRY(cudaEventCreate(&e));
  }
  if (stage != 0 && !((sym || all_tracks) && shard_world > 1))
    return fail(WEALY_ERR_BAD_ARG, "staged runs belong to the sharded all-vs-all sweep");
  if (stage != 2) CU_TRY(cudaEventRecord(p->evs[0], s));
  if (stage != 2) {
    W_TRY(launch_prep(queries_z, ld_q, rows_q, d, dtype, kPrepL2AddEps, eps, pq, nullptr, nullptr, 0, nullptr, 0, s,
                      sym ? p->sorted_idx : nullptr, sym ? (int)nq : 0));
    if (!same) W_TRY(launch_prep(candidates_z, ld_c, rc, d, dtype, kPrepL2AddEps, eps, pc, nullptr, nullptr, 0, nullptr, 0, s));
  }

  // K_pos: relevant similarities, sorted per query
  if (stage != 2) CU_TRY(cudaEventRecord(p->evs[1], s));
  if (stage != 2) {
    const int threads = 256;
    if (sym) {
      // stage 1: this rank's share of the 16-query blocks only; the buffer {lvl, thr} is zeroed first so that the sum
      // over the ranks assembles the whole of it
      int q_lo = 0, q_hi = (int)nq;
      if (stage == 1) {
        const int64_t nblk = ceil_div(nq, 16);
        q_lo = (int)(nblk * shard_rank / shard_world) * 16;
        q_hi = (int)std::min<int64_t>((nblk * (shard_rank + 1) / shard_world) * 16, nq);
        CU_TRY(cudaMemsetAsync(p->lvl_thr_buf, 0, (size_t)p->s_padded * 16 + (size_t)(p->total_pairs > 0 ? p->total_pairs : 1) * 4, s));
      }
      // the plan's cnt array doubles as the per-query fill counter of step 1 (step 2 rewrites it)
      CU_TRY(cudaMemsetAsync(p->cnt, 0, (size_t)nq * 4, s));
      if (q_hi > q_lo)
        pos_pairs_sorted_kernel<false><<<(unsigned)ceil_div(q_hi - q_lo, 16), threads, 0, s>>>(
            pq.hi, pq.lo, (int)pq.d_pad, p->sorted_c, p->s_i, (int)nq, p->s_seg_lo, p->s_seg_len, p->s_off, p->raw, p->cnt, nullptr,
            q_lo, q_hi);
      const unsigned blocks = (unsigned)ceil_div(p->s_padded * 32, threads);
      pos_sort_sorted_kernel<<<blocks, threads, 0, s>>>(p->s_npos, (int)nq, (int)p->s_padded, p->s_off, p->raw, p->thr,
                                                        p->cnt, p->s_lvl, p->s_cinfo, q_lo, q_hi);
    } else if (chunks > 1) {
      // stage 1: this rank's contiguous share of the query tracks, on a zeroed thr (its CSR rows are disjoint from the
      // other ranks', so the sum over the ranks assembles the whole of it); cnt / lim are rebuilt by stage 2
      int q_lo = 0, q_hi = (int)nq;
      if (stage == 1) {
        q_lo = (int)(nq * shard_rank / shard_world);
        q_hi = (int)(nq * (shard_rank + 1) / shard_world);
        CU_TRY(cudaMemsetAsync(p->thr, 0, (size_t)(p->total_pairs > 0 ? p->total_pairs : 1) * 4, s));
      }
      if (q_hi > q_lo)
        pos_thresholds_tracks_kernel<<<(unsigned)(q_hi - q_lo), threads, 0, s>>>(
            pq.hi, pq.lo, pc.hi, pc.lo, (int)pq.d_pad, chunks, red_inner, red_outer, red_scale, p->q_i, (int)nq, p->sorted_idx,
            p->c_i, p->seg_lo, p->seg_len, p->off, p->raw, p->thr, p->lim, p->cnt, q_len, c_len, q_lo);
    } else if (same && p->same_ids && nq > 0 && env_int("WEALY_KPOS_BLOCKS", 1) != 0) {
      // all-vs-all through the rectangle sweep (top-k requested): the clique-block tensor-core K_pos of the symmetric
      // path on the caller's row order (every unordered pair's operands are read once per 16 x 8 block, not per pair)
      CU_TRY(cudaMemsetAsync(p->cnt, 0, (size_t)nq * 4, s));
      pos_pairs_sorted_kernel<true><<<(unsigned)ceil_div(nq, 16), threads, 0, s>>>(
          pq.hi, pq.lo, (int)pq.d_pad, p->sorted_c, p->s_i, (int)nq, p->s_seg_lo, p->s_seg_len, p->off, p->raw, p->cnt,
          p->sorted_idx);
      pos_sort_kernel<<<(unsigned)ceil_div(nq * 32, threads), threads, 0, s>>>((int)nq, p->off, p->raw, p->thr, p->lim, p->cnt);
    } else {
      const unsigned blocks = (unsigned)ceil_div(nq * 32, threads);
      pos_thresholds_kernel<<<blocks, threads, 0, s>>>(pq.hi, pq.lo, pc.hi, pc.lo, (int)pq.d_pad, p->q_i, (int)nq,
                                                       p->sorted_idx, p->c_i, p->seg_lo, p->seg_len, p->off, p->raw,
                                                       p->thr, p->lim, p->cnt);
    }
    CU_TRY(cudaGetLastError());
  }
  if (stage == 1) {
    p->last_sym = sym;
    p->last_stream = s;
    p->staged_chunks = chunks;
    return WEALY_OK;
  }
  if (stage == 2 && chunks > 1) {
    track_limits_kernel<<<(unsigned)ceil_div(nq, 256), 256, 0, s>>>(p->off, p->thr, (int)nq, p->lim, p->cnt);
    CU_TRY(cudaGetLastError());
  }
  // ---- top-k in the symmetric sweep: sampled pre-pass -> per-query lower bound of the k-th best similarity
  float* tk_val = nullptr;
  int *tk_idx = nullptr, *tk_cnt = nullptr, *tk_fail = nullptr;
  float* tk_beta = nullptr;
  int tk_cap2 = 0;
  if (sym_topk) {
    const int n = (int)nq, rows = (int)rows_q;
    // sample ~N/16 rows (>= 4096): the pre-pass is one fp16 pass of N x S pairs.  Target: t = max(24, 3 k S / N) of the
    // sample's similarities above the bound, i.e. about t N / S >= 3 k of the corpus; the bound is the m-th largest of
    // the G = S / 32 group maxima, and the top t of S values occupy about G (1 - exp(-t / G)) distinct groups.
    int S = (int)ceil_div(nq / 16, kTileN) * kTileN;
    if (S < 4096) S = 4096;
    if (S > 32768) S = 32768;
    if (S > n) S = n / kTileN * kTileN;
    const double fr = (double)S / (double)n, G = (double)(S / kChunkCols);
    double t = 3.0 * topk * fr;
    if (t < 24.0) t = 24.0;
    const int r = (int)ceil(G * (1.0 - exp(-t / G)));
    const double mean = t / fr, sd = 1.15 * sqrt(t * (1.0 - fr)) / fr;
    tk_cap2 = (int)align_up((size_t)(mean + 8.0 * sd + 32.0), 32);
    if (tk_cap2 > 1024) tk_cap2 = 1024;
    const int n_groups = S / kChunkCols;
    // carve the scratch
    size_t need_tk = 0;
    auto reserve = [&](size_t bytes) { const size_t o = need_tk; need_tk += align_up(bytes, 1024); return o; };
    const size_t o_samp = reserve((size_t)S * pq.d_pad * 2);
    const size_t o_gmax = reserve((size_t)rows * n_groups * 4);
    const size_t o_beta = reserve((size_t)rows * 4);
    const size_t o_tv = reserve((size_t)rows * tk_cap2 * 4);
    const size_t o_ti = reserve((size_t)rows * tk_cap2 * 4);
    const size_t o_tc = reserve((size_t)rows * 4);
    const size_t o_fail = reserve(256);
    if (need_tk + 1024 > p->tks_cap) {
      big_free(p->tks_buf, p->tks_cap, s);
      p->tks_buf = nullptr;
      p->tks_cap = 0;
      CU_TRY(big_alloc(&p->tks_buf, &p->tks_cap, need_tk + 1024, s));
    }
    uint8_t* tb = reinterpret_cast<uint8_t*>(align_up((size_t)p->tks_buf, 1024));
    __half* samp = reinterpret_cast<__half*>(tb + o_samp);
    float* gmax = reinterpret_cast<float*>(tb + o_gmax);
    tk_beta = reinterpret_cast<float*>(tb + o_beta);
    tk_val = reinterpret_cast<float*>(tb + o_tv);
    tk_idx = reinterpret_cast<int*>(tb + o_ti);
    tk_cnt = reinterpret_cast<int*>(tb + o_tc);
    tk_fail = reinterpret_cast<int*>(tb + o_fail);
    const int T = 256;
    CU_TRY(cudaMemsetAsync(tk_fail, 0, 4, s));
    sample_rows_kernel<<<(unsigned)ceil_div((int64_t)S * 32, T), T, 0, s>>>(pq.hi, (int)pq.d_pad, n, S, samp);
    CU_TRY(cudaGetLastError());
    Planes pa = pq, pb;
    pa.lo = nullptr;
    pb.hi = samp; pb.lo = nullptr; pb.rows = S; pb.d_pad = pq.d_pad;
    pb.norm = pb.scale = pb.sq = nullptr;
    GemmShape shp;
    fill_shape(shp, rows, S, pq.d_pad, 64, 1 << 20, 8);
    GroupMaxParams gp;
    gp.gmax = gmax;
    gp.n_groups = n_groups;
    W_TRY(launch_gemm<GroupMaxEpi>(1, pa, pb, shp, gp, s));  // (the CTA-pair core was measured no faster here: 1.385 vs 1.387 ms for K_pos + pre-pass)
    topk_beta_kernel<<<(unsigned)ceil_div(p->s_padded * 32, 128), 128, 0, s>>>(gmax, n_groups, rows, r + 1, n, tk_beta, p->s_lvl,
                                                                              (int)p->s_padded, tk_cnt);
    CU_TRY(cudaGetLastError());
  }
  p->last_topk_path = topk > 0 ? (sym_topk ? 1 : 2) : 0;
  p->last_sym = sym;
  p->last_stream = s;
  CU_TRY(cudaMemsetAsync(p->hist, 0, (size_t)(p->total_pairs > 0 ? p->total_pairs : 1) * 4, s));
  if (finish) CU_TRY(cudaMemsetAsync(sums, 0, 3 * sizeof(double), s));

  const int halves = 2;  // two epilogue warps per TMEM lane quadrant (16 warps and 4 warps were measured no better)
  GemmShape sh;
  // top-k keeps <= 4 candidate lists per query (column chunks x epilogue warps per row)
  const bool rect_topk = topk > 0 && !sym_topk;
  fill_shape(sh, rq, rc, pq.d_pad, 64, rect_topk ? (4 / halves) : (1 << 20), rect_topk ? 0 : env_int("WEALY_TILES_PER_UNIT", 8));
  const int parts = sh.n_col_chunks * halves;
  const int cap = rect_topk ? topk_capacity(topk) : 0;

  EvalParams ep;
  memset(&ep, 0, sizeof(ep));
  ep.lim = p->lim;
  ep.q_c = p->q_c;
  ep.q_i = p->q_i;
  ep.c_c = p->c_c;
  ep.c_i = p->c_i;
  ep.thr = p->thr;
  ep.off = p->off;
  ep.cnt = p->cnt;
  ep.hist = p->hist;
  ep.topk = topk;
  ep.cap = cap;
  ep.nq_total = (int)nq;
  ep.red_inner = red_inner;
  ep.red_outer = red_outer;
  ep.red_scale = red_scale;
  ep.q_len = q_len;
  ep.c_len = c_len;
  if (rect_topk) {
    const size_t slots = (size_t)parts * nq * cap;
    const size_t tneed = slots * 16 + (size_t)parts * nq * 4 + 1024;  // candidate lists + finalize staging
    if (tneed > p->topk_cap) {
      big_free(p->topk_buf, p->topk_cap, s);
      p->topk_buf = nullptr;
      p->topk_cap = 0;
      CU_TRY(big_alloc((void**)&p->topk_buf, &p->topk_cap, tneed, s));
    }
    ep.cand_val = reinterpret_cast<float*>(p->topk_buf);
    ep.cand_idx = reinterpret_cast<int*>(ep.cand_val + slots);
    ep.cand_cnt = ep.cand_idx + slots;
    CU_TRY(cudaMemsetAsync(ep.cand_cnt, 0, (size_t)parts * nq * 4, s));
  }
  CU_TRY(cudaEventRecord(p->ev0, s));
  // CTA-pair (cta_group::2) kernel: the default for the symmetric sweep (half the B-operand shared-memory traffic;
  // WEALY_SYM_PAIR=0 selects the single-CTA kernel)
  const bool pair = sym && env_int("WEALY_SYM_PAIR", 1) != 0;
  const int total_rb = sh.n_row_blocks;
  if (pair) {
    // the pair kernel works on super row blocks (two adjacent row blocks per CTA pair)
    sh.n_row_blocks = (total_rb + 1) / 2;
    sh.group_rows = (sh.group_rows + 1) / 2;
    // the plain (no top-k) sweep measured best with about half as many super row blocks per scheduling group as there
    // are CTA pairs -- 37 instead of 19 on 148 SMs: 431-443 against 422-436 Gpairs/s at C2 on two boxes (56 .. 74 row
    // blocks the same within the noise, 18 and 296 clearly worse)
    if (!sym_topk && env_int("WEALY_GROUP_ROWS", 0) <= 0) {
      sh.group_rows = std::max(1, num_sms() / 4);
      if (sh.group_rows > sh.n_row_blocks) sh.group_rows = std::max(1, sh.n_row_blocks);
    }
  }
  // (chunked tracks: launch_eval_tracks shards the shape it launches, after halving it into super row blocks)
  if (sym) shard_row_blocks(sh, shard_rank, shard_world);
  if (sym) {
    sh.sym = 1;
    EvalSymParams sp;
    memset(&sp, 0, sizeof(sp));
    sp.lvl = p->s_lvl;
    sp.cinfo = p->s_cinfo;
    sp.s_c = p->sorted_c;
    sp.s_i = p->s_i;
    sp.thr = p->thr;
    sp.hist = p->hist;
    sp.dirty = p->s_dirty;
    sp.n_col_tiles = sh.n_col_tiles;
    sp.n_row_blocks = total_rb;
    sp.total_pairs = (unsigned)p->total_pairs;
    sp.beta = tk_beta;
    sp.tk_val = tk_val;
    sp.tk_idx = tk_idx;
    sp.tk_cnt = tk_cnt;
    sp.tk_cap = tk_cap2;
    const int lv = env_int("WEALY_SYM_LEVELS", 3);  // 3 measured best at C2 (2: 26.8 ms, 3: 25.5 ms, 4: 25.9 ms per step)
    if (sym_topk && pair) {
      // (8 epilogue warps: the top-k epilogue needs 160 registers per thread)
      if (env_int("WEALY_PAIR_INTERLEAVE", 1) != 0) sh.sym |= 2;
      if (passes == 3) {
        sh.k_blocks = (int)(pq.d_pad / 32);
        W_TRY((launch_gemm_pair<EvalSymEpi<3, 256, 4096, true>, 3, 32, 8, true>(pq, sh, sp, s)));
      } else {
        W_TRY((launch_gemm_pair<EvalSymEpi<3, 256, 4096, true>, 1, 64, 8, true>(pq, sh, sp, s)));
      }
    } else if (sym_topk) {
      if (passes == 3) {
        sh.k_blocks = (int)(pq.d_pad / 32);
        W_TRY((launch_gemm_t<EvalSymEpi<3, 256, 4096, true>, 3, 32, 8, 3>(pq, pc, sh, sp, s)));
      } else {
        W_TRY((launch_gemm_t<EvalSymEpi<3, 256, 4096, true>, 1, 64, 8, 3>(pq, pc, sh, sp, s)));
      }
    } else if (pair) {
      if (env_int("WEALY_PAIR_INTERLEAVE", 1) != 0) sh.sym |= 2;
      // three epilogue warps per TMEM lane quadrant (the pair's epilogue is the co-limiter; 16 warps were measured worse);
      // WEALY_PAIR_DYN: the warps of a quadrant claim 32-column chunks dynamically instead of owning fixed ones
      const bool w12 = env_int("WEALY_PAIR_EPI_WARPS", 12) == 12;
      const bool dyn = env_int("WEALY_PAIR_DYN", 1) != 0;
      if (passes == 3) {
        sh.k_blocks = (int)(pq.d_pad / 32);
        // dense threshold levels on the pair core: 4 (C2: 23.45 ms per step against 23.2-23.4 with 3 -- the same --, MAP-0.1
        // data: 43.7 against 49.1 ms; 2 levels: 24.0-24.2 / 56.9 ms)
        const int lvp = env_int("WEALY_SYM_LEVELS", 4);
        if (dyn && w12 && lvp == 2) W_TRY((launch_gemm_pair<EvalSymEpi<2>, 3, 32, 12, true>(pq, sh, sp, s)));
        else if (dyn && w12 && lvp == 4) W_TRY((launch_gemm_pair<EvalSymEpi<4>, 3, 32, 12, true>(pq, sh, sp, s)));
        else if (dyn && w12) W_TRY((launch_gemm_pair<EvalSymEpi<3>, 3, 32, 12, true>(pq, sh, sp, s)));
        else if (dyn) W_TRY((launch_gemm_pair<EvalSymEpi<3>, 3, 32, 8, true>(pq, sh, sp, s)));
        else if (w12) W_TRY((launch_gemm_pair<EvalSymEpi<3>, 3, 32, 12>(pq, sh, sp, s)));
        else W_TRY((launch_gemm_pair<EvalSymEpi<3>, 3, 32>(pq, sh, sp, s)));
      } else {
        if (dyn && w12) W_TRY((launch_gemm_pair<EvalSymEpi<3>, 1, 64, 12, true>(pq, sh, sp, s)));
        else if (dyn) W_TRY((launch_gemm_pair<EvalSymEpi<3>, 1, 64, 8, true>(pq, sh, sp, s)));
        else if (w12) W_TRY((launch_gemm_pair<EvalSymEpi<3>, 1, 64, 12>(pq, sh, sp, s)));
        else W_TRY((launch_gemm_pair<EvalSymEpi<3>, 1, 64>(pq, sh, sp, s)));
      }
    } else if (passes == 3) {
      sh.k_blocks = (int)(pq.d_pad / 32);
      if (lv == 2) W_TRY((launch_gemm_t<EvalSymEpi<2>, 3, 32, 8, 3>(pq, pc, sh, sp, s)));
      else if (lv == 4) W_TRY((launch_gemm_t<EvalSymEpi<4>, 3, 32, 8, 3>(pq, pc, sh, sp, s)));
      else W_TRY((launch_gemm_t<EvalSymEpi<3>, 3, 32, 8, 3>(pq, pc, sh, sp, s)));
    } else {
      W_TRY((launch_gemm_t<EvalSymEpi<3>, 1, 64, 8, 3>(pq, pc, sh, sp, s)));
    }
  } else if (chunks == 2) {
    W_TRY(launch_eval_tracks<2>(passes, pq, pc, sh, ep, s, sym_tracks, shard_rank, shard_world));
  } else if (chunks == 4) {
    W_TRY(launch_eval_tracks<4>(passes, pq, pc, sh, ep, s, sym_tracks, shard_rank, shard_world));
  } else if (chunks == 8) {
    W_TRY(launch_eval_tracks<8>(passes, pq, pc, sh, ep, s, sym_tracks, shard_rank, shard_world));
  } else if (chunks == 16) {
    W_TRY(launch_eval_tracks<16>(passes, pq, pc, sh, ep, s, sym_tracks, shard_rank, shard_world));
  } else {
    W_TRY(launch_gemm_rect<EvalEpi>(passes, pq, pc, sh, ep, s));
  }
  CU_TRY(cudaEventRecord(p->ev1, s));
  p->timed = true;
  p->finished = finish;

  if (local) {
    // (stage events: ap_reduce stays empty -- it runs in wealy_eval_finish once the counters are summed --, topk_finalize
    //  times the local finalize)
    CU_TRY(cudaEventRecord(p->evs[2], s));
    topk_sym_local_kernel<<<(unsigned)ceil_div(rows_q * 32, 128), 128, 0, s>>>(tk_val, tk_idx, tk_cnt, tk_cap2, (int)rows_q, (int)nq,
                                                                              topk, p->sorted_idx, topk_sim, local_idx, local_cnt);
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaEventRecord(p->evs[3], s));
    p->finished = true;
    return WEALY_OK;
  }

  if (finish) {
    const int threads = 256;
    const unsigned blocks = (unsigned)ceil_div(nq * 32, threads);
    if (sym) ap_reduce_kernel<<<blocks, threads, 0, s>>>(p->hist, p->s_off, p->cnt, (int)nq, aps, r1s, sums, p->sorted_idx);
    else ap_reduce_kernel<<<blocks, threads, 0, s>>>(p->hist, p->off, p->cnt, (int)nq, aps, r1s, sums);
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaEventRecord(p->evs[2], s));
    if (sym_topk) {
      topk_sym_finalize_kernel<<<(unsigned)ceil_div(rows_q * 32, 128), 128, 0, s>>>(tk_val, tk_idx, tk_cnt, tk_cap2, (int)rows_q, (int)nq,
                                                                                   topk, p->sorted_idx, (long long*)topk_idx, topk_sim,
                                                                                   tk_fail);
      CU_TRY(cudaGetLastError());
      CU_TRY(cudaEventRecord(p->evs[3], s));
      // the one host round trip of this path: 4 bytes that say whether every list held its k best (see topk_sym_kernels.cuh)
      int failed = 0;
      CU_TRY(cudaMemcpyAsync(&failed, tk_fail, 4, cudaMemcpyDeviceToHost, s));
      CU_TRY(cudaStreamSynchronize(s));
      if (failed != 0) {
        W_TRY(eval_run_impl(p, queries_z, ld_q, candidates_z, ld_c, d, dtype, eps, passes, topk, aps, r1s, sums, topk_idx, topk_sim,
                            shard_rank, shard_world, finish, stream, chunks, redux, q_len, c_len, false));
        p->last_topk_path = 3;
      }
      return WEALY_OK;
    }
    if (topk > 0) {
      if (parts * cap <= 32 * kFinPerLane) {
        float* stage_val = reinterpret_cast<float*>(ep.cand_cnt + (size_t)parts * nq);
        int* stage_idx = reinterpret_cast<int*>(stage_val + (size_t)parts * nq * cap);
        topk_finalize_select_kernel<<<(unsigned)ceil_div(nq * 32, 128), 128, 0, s>>>(
            ep.cand_val, ep.cand_idx, ep.cand_cnt, parts, (int)nq, cap, topk, stage_val, stage_idx,
            (long long*)topk_idx, topk_sim);
      } else {
        topk_finalize_kernel<<<blocks, threads, 0, s>>>(ep.cand_val, ep.cand_idx, ep.cand_cnt, parts, (int)nq, cap, topk,
                                                        (long long*)topk_idx, topk_sim);
      }
      CU_TRY(cudaGetLastError());
    }
    CU_TRY(cudaEventRecord(p->evs[3], s));
  }
  return WEALY_OK;
}

// which kernel produced the top-k lists of the last run: 0 none, 1 symmetric sweep with sampled bounds, 2 rectangle sweep
// (streaming top-k), 3 symmetric sweep whose lists failed the check and were recomputed by the rectangle sweep
extern "C" int wealy_eval_plan_last_topk_path(const wealy_eval_plan* p, int* path) {
  if (!p || !path) return fail(WEALY_ERR_BAD_ARG, "null pointer");
  *path = p->last_topk_path;
  return WEALY_OK;
}

// device time of the stages of the last run: {prep, K_pos (+ counter reset), fused sweep, ap_reduce, top-k finalize}
extern "C" int wealy_eval_plan_stage_ms(const wealy_eval_plan* p, float* ms) {
  if (!p || !ms) return fail(WEALY_ERR_BAD_ARG, "null pointer");
  if (!p->timed) return fail(WEALY_ERR_BAD_ARG, "the plan has not been run yet");
  CU_TRY(cudaEventSynchronize(p->finished ? p->evs[3] : p->ev1));
  CU_TRY(cudaEventElapsedTime(&ms[0], p->evs[0], p->evs[1]));
  CU_TRY(cudaEventElapsedTime(&ms[1], p->evs[1], p->ev0));
  CU_TRY(cudaEventElapsedTime(&ms[2], p->ev0, p->ev1));
  ms[3] = ms[4] = 0.f;
  if (p->finished) {
    CU_TRY(cudaEventElapsedTime(&ms[3], p->ev1, p->evs[2]));
    CU_TRY(cudaEventElapsedTime(&ms[4], p->evs[2], p->evs[3]));
  }
  return WEALY_OK;
}

extern "C" int wealy_eval_run(wealy_eval_plan* p, const void* queries_z, int64_t ld_q, const void* candidates_z,
                              int64_t ld_c, int64_t d, int dtype, float eps, int passes, int topk, float* aps,
                              float* r1s, double* sums, int64_t* topk_idx, float* topk_sim, void* stream) {
  return eval_run_impl(p, queries_z, ld_q, candidates_z, ld_c, d, dtype, eps, passes, topk, aps, r1s, sums, topk_idx,
                       topk_sim, 0, 1, true, stream);
}

// ------------------------------------------------------------------------------------------
// All-vs-all evaluation of embeddings that still live in PINNED HOST memory: upload, normalisation and the symmetric
// sweep as one pipeline.  The sweep runs in the plan's clique-sorted row order and a super row block only needs the
// rows BEHIND it (tiles above the diagonal), so the rows are fetched from the end: part by part a small persistent
// kernel (prep_rows_stream_kernel, on its own stream and on a few SMs of its own) reads the caller's rows over
// PCIe in sorted order -- a gather no copy engine can do --, and as soon as a part has arrived its relevant
// similarities (K_pos) and its row blocks of the sweep run on the caller's stream while the next part is in flight.
// Parts grow towards the front: the work of a part grows with the square of the rows behind it.
// ------------------------------------------------------------------------------------------
static cudaStream_t upload_stream() {
  static cudaStream_t streams[64] = {nullptr};
  static std::mutex mu;
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64) return nullptr;
  std::lock_guard<std::mutex> lock(mu);
  if (!streams[dev] && cudaStreamCreateWithFlags(&streams[dev], cudaStreamNonBlocking) != cudaSuccess) streams[dev] = nullptr;
  return streams[dev];
}

template <int kLevels, int kPasses, int kBlockK>
static int launch_sym_part(const Planes& pq, const GemmShape& sh, const EvalSymParams& sp, cudaStream_t s, int max_pairs) {
  return launch_gemm_pair<EvalSymEpi<kLevels>, kPasses, kBlockK, 12, true>(pq, sh, sp, s, nullptr, max_pairs);
}

// The upload kernel and where it runs.  By default on U = 8 SMs of its own (WEALY_HOST_UP_SMS): CTAs of 512 threads whose
// shared-memory request keeps the sweep off their SM, while the parts of the sweep that can overlap with the upload run
// on the remaining SMs.  Measured at 100 000 x 1024 (profiles/r02_host_pipeline.md): 8 SMs already saturate PCIe
// (51 GB/s).  U = 0 puts two upload warps per SM NEXT to the sweep's CTAs (they fit beside a resident sweep CTA; the
// largest shared-memory carve-out is requested for them and for the K_pos kernels between the parts, because an SM whose
// L1 / shared-memory split was chosen for a kernel without shared memory cannot take a sweep CTA until it has drained):
// that slowed the sweep and K_pos 2-3x while rows were in flight -- the SM's memory pipeline queues behind the
// microsecond-long host reads.  K_pos also slows down with the number of SMs that read host memory (U = 4: not at all,
// U = 16: 4x).
struct HostUpload {
  const void* z = nullptr;  // device-side address of the pinned host matrix
  int64_t ld = 0, d = 0;
  int dtype = 0;
  float eps = 0.f;
  int up_sms = 0, grid = 0, threads = 0;
  size_t smem = 0;
  cudaStream_t up = nullptr;
};

// status: WEALY_OK, or why the device cannot read these embeddings (*on_device: a device pointer, take the plain path)
static int host_upload_setup(HostUpload& h, const void* host_z, int64_t ld, int64_t d, int dtype, float eps, bool* on_device) {
  *on_device = false;
  if (dtype != WEALY_F32 && dtype != WEALY_F16 && dtype != WEALY_BF16) return fail(WEALY_ERR_BAD_ARG, "unknown element type %d", dtype);
  cudaPointerAttributes attr;
  if (cudaPointerGetAttributes(&attr, host_z) != cudaSuccess) {
    cudaGetLastError();
    return fail(WEALY_ERR_UNSUPPORTED, "cannot classify the embeddings' pointer");
  }
  if (attr.type == cudaMemoryTypeDevice || attr.type == cudaMemoryTypeManaged) {
    *on_device = true;
    return WEALY_OK;
  }
  if (d <= 0 || d > 128 * kRowVecs || d % 4 != 0 || ld % 4 != 0 || ld < d)
    return fail(WEALY_ERR_UNSUPPORTED, "wealy_eval_run_host needs rows of 4 k <= %d elements (d=%lld, ld=%lld)", 128 * kRowVecs,
                (long long)d, (long long)ld);
  if (attr.type != cudaMemoryTypeHost || !attr.devicePointer)
    return fail(WEALY_ERR_UNSUPPORTED, "host embeddings must be pinned (page-locked and mapped) to be read by the device");
  h.z = attr.devicePointer;
  if ((reinterpret_cast<uintptr_t>(h.z) & 15) != 0) return fail(WEALY_ERR_UNSUPPORTED, "host embeddings must be 16-byte aligned");
  h.ld = ld;
  h.d = d;
  h.dtype = dtype;
  h.eps = eps;
  h.up = upload_stream();
  if (!h.up) return fail(WEALY_ERR_CUDA, "no upload stream");
  h.up_sms = std::min(std::max(env_int("WEALY_HOST_UP_SMS", 8), 0), num_sms() / 2);
  h.smem = h.up_sms > 0 ? 120 * 1024 : 0;
  h.grid = h.up_sms > 0 ? h.up_sms : num_sms() * std::max(1, env_int("WEALY_HOST_UP_GRID", 1));
  if (h.up_sms > 0) {
    h.threads = std::min(512, std::max(32, env_int("WEALY_HOST_UP_THREADS", 512) / 32 * 32));  // (bytes in flight per upload SM)
  } else {
    h.threads = env_int("WEALY_HOST_UP_THREADS", 64) <= 32 ? 32 : 64;
  }
  const void* up_kernel =
      h.up_sms > 0 ? (dtype == WEALY_F32 ? (const void*)prep_rows_stream_kernel<float, 512>
                      : dtype == WEALY_F16 ? (const void*)prep_rows_stream_kernel<__half, 512>
                                           : (const void*)prep_rows_stream_kernel<__nv_bfloat16, 512>)
                   : (dtype == WEALY_F32 ? (const void*)prep_rows_stream_kernel<float, 64>
                      : dtype == WEALY_F16 ? (const void*)prep_rows_stream_kernel<__half, 64>
                                           : (const void*)prep_rows_stream_kernel<__nv_bfloat16, 64>);
  CU_TRY(cudaFuncSetAttribute(up_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  if (h.smem) CU_TRY(cudaFuncSetAttribute(up_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h.smem));
  return WEALY_OK;
}

// plane rows [lo, hi) (whole 128-row blocks of the spread order) <- the caller's rows, on the upload stream
static int host_upload_rows(const HostUpload& h, const Planes& pq, const int* sorted_idx, int64_t n, int64_t lo, int64_t hi) {
  if (hi <= lo) return WEALY_OK;
#define STREAM_ARGS (long long)h.ld, (int)lo, (int)hi, (int)h.d, (int)pq.d_pad, h.eps, pq.hi, pq.lo, pq.norm, pq.scale, pq.sq, sorted_idx, (int)n
#define STREAM_LAUNCH(T)                                                                                                     \
  do {                                                                                                                       \
    if (h.up_sms > 0) prep_rows_stream_kernel<T, 512><<<h.grid, h.threads, h.smem, h.up>>>((const T*)h.z, STREAM_ARGS);       \
    else prep_rows_stream_kernel<T, 64><<<h.grid, h.threads, 0, h.up>>>((const T*)h.z, STREAM_ARGS);                          \
  } while (0)
  switch (h.dtype) {
    case WEALY_F32: STREAM_LAUNCH(float); break;
    case WEALY_F16: STREAM_LAUNCH(__half); break;
    default: STREAM_LAUNCH(__nv_bfloat16); break;
  }
#undef STREAM_LAUNCH
#undef STREAM_ARGS
  CU_TRY(cudaGetLastError());
  return WEALY_OK;
}

// operand planes of an all-vs-all plan in the sweep's spread order over whole 128-row blocks, and the events of a host run
static int host_planes(wealy_eval_plan* p, int64_t d, int passes, cudaStream_t s, Planes& pq) {
  const int64_t rows_q = ceil_div(p->nq, kTileM) * kTileM;
  const size_t need = planes_bytes(rows_q, d, passes) + 2048;
  if (need > p->planes_cap) {
    big_free(p->planes_buf, p->planes_cap, s);
    p->planes_buf = nullptr;
    p->planes_cap = 0;
    CU_TRY(big_alloc((void**)&p->planes_buf, &p->planes_cap, need, s));
  }
  uint8_t* cur = reinterpret_cast<uint8_t*>(align_up((size_t)p->planes_buf, 1024));
  carve_planes(pq, cur, rows_q, d, passes);
  if (!p->ev0) {
    CU_TRY(cudaEventCreate(&p->ev0));
    CU_TRY(cudaEventCreate(&p->ev1));
    for (cudaEvent_t& e : p->evs) CU_TRY(cudaEventCreate(&e));
  }
  for (cudaEvent_t& e : p->host_ev)
    if (!e) CU_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  return WEALY_OK;
}

// parts of a host run, in super row blocks (256 rows) counted from the END: cumulative fractions of the rows
static float kHostCum[5][8] = {{1.f}, {0.30f, 1.f}, {0.10f, 0.20f, 0.35f, 0.55f, 1.f}, {0.06f, 0.14f, 0.24f, 0.36f, 0.5f, 0.7f, 1.f}, {1.f}};
static int kHostCount[5] = {1, 2, 5, 7, 1};
static int host_preset(int64_t n) {
  const int nsb = (int)ceil_div(n, 2 * kTileM);
  int preset = nsb >= 96 ? 2 : (nsb >= 24 ? 1 : 0);  // (24 k / 6 k rows)
  const int forced = env_int("WEALY_HOST_PARTS", 0);
  if (forced > 0) preset = forced >= 7 ? 3 : (forced >= 5 ? 2 : (forced >= 2 ? 1 : 0));
  // WEALY_HOST_CUM="0.1,0.25,0.5" (tuning): a schedule of its own, up to 7 increasing fractions; 1.0 is appended
  if (const char* cum = getenv("WEALY_HOST_CUM")) {
    static std::mutex mu;
    std::lock_guard<std::mutex> lock(mu);
    int cnt = 0;
    float last = 0.f;
    for (const char* q = cum; *q && cnt < 7;) {
      char* end = nullptr;
      const float v = strtof(q, &end);
      if (end == q) break;
      if (v > last && v < 1.f) kHostCum[4][cnt++] = last = v;
      q = *end == ',' ? end + 1 : end;
      if (*end != ',' && *end != 0) break;
    }
    kHostCum[4][cnt++] = 1.f;
    kHostCount[4] = cnt;
    preset = 4;
  }
  return preset;
}
// first super row block of part k
static int host_part_begin(int64_t n, int preset, int k) {
  const int nsb = (int)ceil_div(n, 2 * kTileM);
  if (k + 1 >= kHostCount[preset]) return 0;
  const int sb = nsb - (int)lroundf(kHostCum[preset][k] * (float)nsb);
  return sb < 0 ? 0 : sb;
}

// As wealy_eval_plan_create for an all-vs-all evaluation of pinned host embeddings (to be run with wealy_eval_run_host on
// the same matrix): the upload of the first part starts as soon as the sorted order exists, under the rest of the plan.
extern "C" int wealy_eval_plan_create_host(const int64_t* queries_c, const int64_t* queries_i, int64_t nq,
                                           const int64_t* candidates_c, const int64_t* candidates_i, int64_t nc,
                                           const void* host_z, int64_t ld, int64_t d, int dtype, float eps, int passes,
                                           void* stream, wealy_eval_plan** plan) {
  if (!plan) return fail(WEALY_ERR_BAD_ARG, "plan output pointer is null");
  *plan = nullptr;
  if (nq <= 0 || nc <= 0) return fail(WEALY_ERR_BAD_ARG, "empty query or candidate set (nq=%lld nc=%lld)", (long long)nq, (long long)nc);
  if (!queries_c || !queries_i || !candidates_c || !candidates_i) return fail(WEALY_ERR_BAD_ARG, "null id pointer");
  if (nq >= (1ll << 31) - 256 || nc >= (1ll << 31) - 256) return fail(WEALY_ERR_UNSUPPORTED, "more than 2^31 rows");
  cudaStream_t s = (cudaStream_t)stream;
  wealy_eval_plan* p = new wealy_eval_plan();
  p->nq = nq;
  p->nc = nc;
  p->stream = s;
  auto early = [&]() -> int {
    HostUpload h;
    bool on_device = false;
    if (!host_z || (passes != 1 && passes != 3) || env_int("WEALY_HOST_EARLY", 1) == 0) return WEALY_OK;
    if (host_upload_setup(h, host_z, ld, d, dtype, eps, &on_device) != WEALY_OK || on_device) return WEALY_OK;  // nothing to start early
    Planes pq;
    W_TRY(host_planes(p, d, passes, s, pq));
    const int64_t lo = (int64_t)host_part_begin(nq, host_preset(nq), 0) * 2 * kTileM;
    CU_TRY(cudaEventRecord(p->host_ev[0], s));
    CU_TRY(cudaStreamWaitEvent(h.up, p->host_ev[0], 0));
    W_TRY(host_upload_rows(h, pq, p->sorted_idx, nq, lo, pq.rows));
    p->early_lo = lo;
    p->early_z = h.z;
    p->early_ld = ld;
    p->early_d = d;
    p->early_dtype = dtype;
    p->early_passes = passes;
    p->early_eps = eps;
    return WEALY_OK;
  };
  int st = plan_build(p, queries_c, queries_i, candidates_c, candidates_i, s, early);
  if (st != WEALY_OK) {
    wealy_eval_plan_destroy(p);
    return st;
  }
  *plan = p;
  return WEALY_OK;
}

extern "C" int wealy_eval_run_host(wealy_eval_plan* p, const void* host_z, int64_t ld, int64_t d, int dtype, float eps,
                                   int passes, float* aps, float* r1s, double* sums, void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  if (!p || !host_z || !aps || !r1s || !sums) return fail(WEALY_ERR_BAD_ARG, "null pointer");
  if (passes != 1 && passes != 3) return fail(WEALY_ERR_BAD_ARG, "passes must be 1 or 3");
  const int64_t n = p->nq;
  if (!(p->same_ids && p->nq == p->nc && p->total_pairs < (1ll << 31) - 8))
    return fail(WEALY_ERR_UNSUPPORTED, "wealy_eval_run_host evaluates all-vs-all plans (queries == candidates)");
  HostUpload h;
  bool on_device = false;
  W_TRY(host_upload_setup(h, host_z, ld, d, dtype, eps, &on_device));
  if (on_device)  // already on the device: the plain run
    return eval_run_impl(p, host_z, ld, host_z, ld, d, dtype, eps, passes, 0, aps, r1s, sums, nullptr, nullptr, 0, 1, true, stream);
  const void* z = h.z;
  cudaStream_t up = h.up;
  const int up_sms = h.up_sms;
  const void* kpos_kernels[2] = {(const void*)pos_pairs_sorted_kernel<false>, (const void*)pos_sort_sorted_kernel};
  struct RestoreCarveout {
    const void* const* k;
    bool on;
    ~RestoreCarveout() {
      for (int i = 0; on && i < 2; ++i) cudaFuncSetAttribute(k[i], cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutDefault);
    }
  } restore{kpos_kernels, up_sms == 0};
  if (up_sms == 0)  // (upload CTAs on SMs of their own never share an SM with these kernels; the attribute is read at launch)
    for (const void* k : kpos_kernels)
      CU_TRY(cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));

  Planes pq;
  W_TRY(host_planes(p, d, passes, s, pq));
  const int64_t rows_q = pq.rows;
  // rows an early upload (wealy_eval_plan_create_host) of exactly this matrix has already put in flight
  int64_t early_lo = -1;
  if (p->early_lo >= 0 && p->early_z == z && p->early_ld == ld && p->early_d == d && p->early_dtype == dtype &&
      p->early_passes == passes && p->early_eps == eps)
    early_lo = p->early_lo;
  p->early_lo = -1;

  const int nsb = (int)ceil_div(n, 2 * kTileM);
  const int preset = host_preset(n);
  const int n_parts = kHostCount[preset];
  const int64_t reach = p->max_clique > 1 ? p->max_clique : 1;  // K_pos of a query reads the rows of its whole clique

  GemmShape sh0;
  fill_shape(sh0, n, n, pq.d_pad, 64, 1 << 20, env_int("WEALY_TILES_PER_UNIT", 8));
  const int total_rb = sh0.n_row_blocks;
  sh0.sym = 1 | (env_int("WEALY_PAIR_INTERLEAVE", 1) != 0 ? 2 : 0);
  if (passes == 3) sh0.k_blocks = (int)(pq.d_pad / 32);
  EvalSymParams sp;
  memset(&sp, 0, sizeof(sp));
  sp.lvl = p->s_lvl;
  sp.cinfo = p->s_cinfo;
  sp.s_c = p->sorted_c;
  sp.s_i = p->s_i;
  sp.thr = p->thr;
  sp.hist = p->hist;
  sp.dirty = p->s_dirty;
  sp.n_col_tiles = sh0.n_col_tiles;
  sp.n_row_blocks = total_rb;
  sp.total_pairs = (unsigned)p->total_pairs;

  CU_TRY(cudaEventRecord(p->evs[0], s));
  CU_TRY(cudaEventRecord(p->evs[1], s));
  CU_TRY(cudaMemsetAsync(p->hist, 0, (size_t)(p->total_pairs > 0 ? p->total_pairs : 1) * 4, s));
  CU_TRY(cudaMemsetAsync(p->cnt, 0, (size_t)n * 4, s));
  CU_TRY(cudaMemsetAsync(sums, 0, 3 * sizeof(double), s));
  CU_TRY(cudaEventRecord(p->host_ev[0], s));           // the upload may touch the planes from here on
  CU_TRY(cudaStreamWaitEvent(up, p->host_ev[0], 0));
  CU_TRY(cudaEventRecord(p->ev0, s));

  // WEALY_HOST_TRACE=1 (diagnostics): time stamps of every part on both streams, printed to stderr after a synchronize
  const bool trace = env_int("WEALY_HOST_TRACE", 0) != 0;
  std::vector<cudaEvent_t> tev;
  auto stamp = [&](cudaStream_t st) {
    if (!trace) return;
    cudaEvent_t e = nullptr;
    cudaEventCreate(&e);
    cudaEventRecord(e, st);
    tev.push_back(e);
  };
  stamp(s);
  int sb_hi = nsb;
  int64_t prep_hi = rows_q;
  for (int k = 0; k < n_parts; ++k) {
    int sb_lo = host_part_begin(n, preset, k);
    if (sb_lo > sb_hi) sb_lo = sb_hi;
    // ---- upload stream: the rows this part's sweep AND its K_pos need (its cliques may start `reach` rows earlier)
    int64_t prep_lo = k + 1 == n_parts ? 0 : ((int64_t)sb_lo * 2 * kTileM - reach) / kTileM * kTileM;
    if (prep_lo < 0) prep_lo = 0;
    if (prep_lo > prep_hi) prep_lo = prep_hi;
    stamp(up);
    // (what an early upload already has in flight is not fetched again)
    W_TRY(host_upload_rows(h, pq, p->sorted_idx, n, prep_lo, early_lo >= 0 ? std::min(prep_hi, early_lo) : prep_hi));
    if (trace) fprintf(stderr, "[wealy host run] part %d: rows [%lld, %lld) arrive, super row blocks [%d, %d) swept\n", k,
                       (long long)prep_lo, (long long)prep_hi, sb_lo, sb_hi);
    prep_hi = prep_lo;
    stamp(up);
    CU_TRY(cudaEventRecord(p->host_ev[1 + k], up));
    CU_TRY(cudaStreamWaitEvent(s, p->host_ev[1 + k], 0));
    stamp(s);
    // ---- caller's stream: K_pos of the part's queries, then its row blocks of the sweep
    const int q_lo = sb_lo * 2 * kTileM;
    const int q_hi = (int)std::min<int64_t>((int64_t)sb_hi * 2 * kTileM, n);
    if (q_hi > q_lo) {
      const int threads = 256;
      pos_pairs_sorted_kernel<false><<<(unsigned)ceil_div(q_hi - q_lo, 16), threads, 0, s>>>(
          pq.hi, pq.lo, (int)pq.d_pad, p->sorted_c, p->s_i, (int)n, p->s_seg_lo, p->s_seg_len, p->s_off, p->raw, p->cnt, nullptr,
          q_lo, q_hi);
      const int64_t sort_end = k == 0 ? p->s_padded : q_hi;  // (the first part reaches n: it owns the padding rows)
      pos_sort_sorted_kernel<<<(unsigned)ceil_div((sort_end - q_lo) * 32, threads), threads, 0, s>>>(
          p->s_npos, (int)n, (int)p->s_padded, p->s_off, p->raw, p->thr, p->cnt, p->s_lvl, p->s_cinfo, q_lo, q_hi, 1);
      CU_TRY(cudaGetLastError());
      stamp(s);
      GemmShape sh = sh0;
      sh.n_row_blocks = sb_hi - sb_lo;
      sh.rb_offset = sb_lo;
      sh.rb_stride = 1;
      sh.group_rows = std::max(1, std::min(num_sms() / 4, sh.n_row_blocks));
      const int max_pairs = (up_sms > 0 && k + 1 < n_parts) ? (num_sms() - up_sms) / 2 : 0;
      if (passes == 3) W_TRY((launch_sym_part<4, 3, 32>(pq, sh, sp, s, max_pairs)));
      else W_TRY((launch_sym_part<3, 1, 64>(pq, sh, sp, s, max_pairs)));
    }
    else stamp(s);
    stamp(s);
    sb_hi = sb_lo;
  }
  CU_TRY(cudaEventRecord(p->ev1, s));
  if (trace) {
    cudaStreamSynchronize(s);
    cudaStreamSynchronize(up);
    // per part: {upload begin, upload end} on the upload stream, {wait over, K_pos done, sweep done} on the run's stream
    for (int k = 0; k < n_parts && (size_t)(1 + 5 * k + 4) < tev.size(); ++k) {
      float t[5];
      for (int j = 0; j < 5; ++j) cudaEventElapsedTime(&t[j], tev[0], tev[1 + 5 * k + j]);
      fprintf(stderr, "[wealy host run] part %d: upload %.3f -> %.3f ms | ready %.3f, K_pos done %.3f, sweep done %.3f ms\n", k, t[0],
              t[1], t[2], t[3], t[4]);
    }
    for (cudaEvent_t e : tev) cudaEventDestroy(e);
  }
  p->timed = true;
  p->finished = true;
  p->last_sym = true;
  p->last_stream = s;
  p->last_topk_path = 0;
  ap_reduce_kernel<<<(unsigned)ceil_div(n * 32, 256), 256, 0, s>>>(p->hist, p->s_off, p->cnt, (int)n, aps, r1s, sums, p->sorted_idx);
  CU_TRY(cudaGetLastError());
  CU_TRY(cudaEventRecord(p->evs[2], s));
  CU_TRY(cudaEventRecord(p->evs[3], s));
  return WEALY_OK;
}

extern "C" int wealy_eval_run_chunked(wealy_eval_plan* p, const void* queries_z, int64_t ld_q, const void* candidates_z,
                                      int64_t ld_c, int64_t d, int dtype, float eps, int passes, int topk, int chunks,
                                      int redux, float* aps, float* r1s, double* sums, int64_t* topk_idx, float* topk_sim,
                                      void* stream) {
  return eval_run_impl(p, queries_z, ld_q, candidates_z, ld_c, d, dtype, eps, passes, topk, aps, r1s, sums, topk_idx,
                       topk_sim, 0, 1, true, stream, chunks, redux);
}

extern "C" int wealy_eval_run_ragged(wealy_eval_plan* p, const void* queries_z, int64_t ld_q, const void* candidates_z,
                                     int64_t ld_c, int64_t d, int dtype, float eps, int passes, int topk, int chunks,
                                     int redux, const int32_t* q_len, const int32_t* c_len, float* aps, float* r1s,
                                     double* sums, int64_t* topk_idx, float* topk_sim, void* stream) {
  if (!q_len || !c_len) return fail(WEALY_ERR_BAD_ARG, "null chunk counts");
  return eval_run_impl(p, queries_z, ld_q, candidates_z, ld_c, d, dtype, eps, passes, topk, aps, r1s, sums, topk_idx,
                       topk_sim, 0, 1, true, stream, chunks, redux, q_len, c_len);
}

// The same in two stages, so that the relevant similarities (K_pos) are computed ONCE across the ranks instead of once
// per rank: _prepare preps the planes and fills this rank's share of the threshold buffer (zeros elsewhere), the caller
// sums the buffer of wealy_eval_plan_thresholds over the ranks (one all-reduce of floats), _sweep runs the rank's
// share of the row blocks on the result.
extern "C" int wealy_eval_shard_prepare(wealy_eval_plan* p, const void* z, int64_t ld, int64_t d, int dtype, float eps,
                                        int passes, int shard_rank, int shard_world, void* stream) {
  if (shard_world < 2) return fail(WEALY_ERR_BAD_ARG, "staged sweeps are for two or more ranks");
  return eval_run_impl(p, z, ld, z, ld, d, dtype, eps, passes, 0, nullptr, nullptr, nullptr, nullptr, nullptr, shard_rank,
                       shard_world, false, stream, 1, WEALY_REDUX_MIN, nullptr, nullptr, true, 1);
}

extern "C" int wealy_eval_plan_thresholds(const wealy_eval_plan* p, void** values, int64_t* count) {
  if (!p || !values || !count) return fail(WEALY_ERR_BAD_ARG, "null pointer");
  if (!p->lvl_thr_buf) return fail(WEALY_ERR_BAD_ARG, "the plan is not an all-vs-all plan");
  if (p->staged_chunks > 1) {  // chunked tracks: the thresholds in the caller's CSR order, nothing else
    *values = p->thr;
    *count = p->total_pairs > 0 ? p->total_pairs : 1;
    return WEALY_OK;
  }
  *values = p->lvl_thr_buf;
  *count = p->s_padded * 4 + (p->total_pairs > 0 ? p->total_pairs : 1);
  return WEALY_OK;
}

// Chunked tracks (chunks in {2, 4, 8, 16}, redux WEALY_REDUX_*, lens = NULL or the ragged chunk counts of every track):
// the same three steps.  min / max / mean take the half sweep, the other reductions (and small sets, WEALY_SYM_TRACKS=0)
// the rectangle sweep; either way sharded by row blocks.
static int check_shard_tracks(const wealy_eval_plan* p, int chunks, int shard_rank, int shard_world) {
  if (!p) return fail(WEALY_ERR_BAD_ARG, "null plan");
  if (!p->same_ids) return fail(WEALY_ERR_BAD_ARG, "a sharded sweep needs queries == candidates (ids and embeddings) and no top-k");
  if (chunks != 2 && chunks != 4 && chunks != 8 && chunks != 16)
    return fail(WEALY_ERR_UNSUPPORTED, "chunked tracks have 2, 4, 8 or 16 chunks, got %d", chunks);
  if (shard_world < 1 || shard_rank < 0 || shard_rank >= shard_world) return fail(WEALY_ERR_BAD_ARG, "bad shard %d/%d", shard_rank, shard_world);
  return WEALY_OK;
}

extern "C" int wealy_eval_sweep_shard_tracks(wealy_eval_plan* p, const void* z, int64_t ld, int64_t d, int dtype, float eps,
                                             int passes, int chunks, int redux, const int32_t* lens, int shard_rank,
                                             int shard_world, void* stream) {
  W_TRY(check_shard_tracks(p, chunks, shard_rank, shard_world));
  return eval_run_impl(p, z, ld, z, ld, d, dtype, eps, passes, 0, nullptr, nullptr, nullptr, nullptr, nullptr, shard_rank,
                       shard_world, false, stream, chunks, redux, lens, lens);
}

extern "C" int wealy_eval_shard_prepare_tracks(wealy_eval_plan* p, const void* z, int64_t ld, int64_t d, int dtype, float eps,
                                               int passes, int chunks, int redux, const int32_t* lens, int shard_rank,
                                               int shard_world, void* stream) {
  W_TRY(check_shard_tracks(p, chunks, shard_rank, shard_world));
  if (shard_world < 2) return fail(WEALY_ERR_BAD_ARG, "staged sweeps are for two or more ranks");
  return eval_run_impl(p, z, ld, z, ld, d, dtype, eps, passes, 0, nullptr, nullptr, nullptr, nullptr, nullptr, shard_rank,
                       shard_world, false, stream, chunks, redux, lens, lens, true, 1);
}

extern "C" int wealy_eval_shard_sweep_tracks(wealy_eval_plan* p, int64_t d, int passes, int chunks, int redux,
                                             const int32_t* lens, int shard_rank, int shard_world, void* stream) {
  W_TRY(check_shard_tracks(p, chunks, shard_rank, shard_world));
  if (shard_world < 2) return fail(WEALY_ERR_BAD_ARG, "staged sweeps are for two or more ranks");
  return eval_run_impl(p, nullptr, 0, nullptr, 0, d, WEALY_F32, 0.f, passes, 0, nullptr, nullptr, nullptr, nullptr, nullptr,
                       shard_rank, shard_world, false, stream, chunks, redux, lens, lens, true, 2);
}

extern "C" int wealy_eval_shard_sweep(wealy_eval_plan* p, int64_t d, int passes, int shard_rank, int shard_world, void* stream) {
  if (shard_world < 2) return fail(WEALY_ERR_BAD_ARG, "staged sweeps are for two or more ranks");
  return eval_run_impl(p, nullptr, 0, nullptr, 0, d, WEALY_F32, 0.f, passes, 0, nullptr, nullptr, nullptr, nullptr, nullptr,
                       shard_rank, shard_world, false, stream, 1, WEALY_REDUX_MIN, nullptr, nullptr, true, 2);
}

// multi-GPU all-vs-all: every rank sweeps its share of the row blocks of the SAME symmetric problem ...
extern "C" int wealy_eval_sweep_shard(wealy_eval_plan* p, const void* z, int64_t ld, int64_t d, int dtype, float eps,
                                      int passes, int shard_rank, int shard_world, void* stream) {
  return eval_run_impl(p, z, ld, z, ld, d, dtype, eps, passes, 0, nullptr, nullptr, nullptr, nullptr, nullptr,
                       shard_rank, shard_world, false, stream);
}

// ... with top-k lists: the same sweep with the symmetric top-k epilogue, this rank's lists finalized locally (caller's
// row order; cnt -1 = overflow); eligibility depends on the arguments and the plan's ids only, so every rank gets the
// same answer before any work.  world * k <= 1024: the merge takes a query's lists of all ranks in one warp pass.
extern "C" int wealy_eval_sweep_shard_topk(wealy_eval_plan* p, const void* z, int64_t ld, int64_t d, int dtype, float eps,
                                           int passes, int k, int shard_rank, int shard_world, float* val, int32_t* idx,
                                           int32_t* cnt, void* stream) {
  if (k < 1 || k > 128) return fail(WEALY_ERR_UNSUPPORTED, "the sharded top-k sweep needs 1 <= k <= 128, got %d", k);
  if ((int64_t)shard_world * k > 1024)
    return fail(WEALY_ERR_UNSUPPORTED, "the sharded top-k merge needs world * k <= 1024, got %d x %d", shard_world, k);
  if (!p || !z || !val || !idx || !cnt) return fail(WEALY_ERR_BAD_ARG, "null pointer");
  return eval_run_impl(p, z, ld, z, ld, d, dtype, eps, passes, k, nullptr, nullptr, nullptr, nullptr, val, shard_rank,
                       shard_world, false, stream, 1, WEALY_REDUX_MIN, nullptr, nullptr, true, 0, idx, cnt);
}

// The k best of every query's lists of all ranks (val / idx [world][n][k], cnt [world][n]: the local lists of the ranks,
// each restricted to the same n queries) -> out_idx / out_sim [n][k]; *fail += the queries whose lists overflowed or
// hold fewer than k entries together.
extern "C" int wealy_eval_topk_merge(const float* val, const int32_t* idx, const int32_t* cnt, int world, int64_t n, int k,
                                     int64_t* out_idx, float* out_sim, int32_t* fail_count, void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  if (world < 1 || n < 0 || k < 1) return fail(WEALY_ERR_BAD_ARG, "bad merge shape: %d lists of [%lld][%d]", world, (long long)n, k);
  if (k > 128 || (int64_t)world * k > 1024)
    return fail(WEALY_ERR_UNSUPPORTED, "the top-k merge needs k <= 128 and world * k <= 1024, got %d x %d", world, k);
  if (n == 0) return WEALY_OK;
  if (!val || !idx || !cnt || !out_idx || !out_sim || !fail_count) return fail(WEALY_ERR_BAD_ARG, "null pointer");
  const unsigned blocks = (unsigned)ceil_div(n * 32, 128);
  const int L = world * k;
  long long* oi = reinterpret_cast<long long*>(out_idx);
  if (L <= 128) topk_merge_kernel<4><<<blocks, 128, 0, s>>>(val, idx, cnt, world, n, k, oi, out_sim, fail_count);
  else if (L <= 256) topk_merge_kernel<8><<<blocks, 128, 0, s>>>(val, idx, cnt, world, n, k, oi, out_sim, fail_count);
  else if (L <= 512) topk_merge_kernel<16><<<blocks, 128, 0, s>>>(val, idx, cnt, world, n, k, oi, out_sim, fail_count);
  else topk_merge_kernel<32><<<blocks, 128, 0, s>>>(val, idx, cnt, world, n, k, oi, out_sim, fail_count);
  CU_TRY(cudaGetLastError());
  return WEALY_OK;
}

// ... the per-(query, relevant item) rank counts are then summed over the ranks by the caller (an all-reduce of
// `count` uint32 values starting at `counts`) ...
extern "C" int wealy_eval_plan_counts(const wealy_eval_plan* p, void** counts, int64_t* count) {
  if (!p || !counts || !count) return fail(WEALY_ERR_BAD_ARG, "null pointer");
  *counts = p->hist;
  *count = p->total_pairs > 0 ? p->total_pairs : 1;
  return WEALY_OK;
}

// ... and turned into AP / R1 / sums on every rank.
extern "C" int wealy_eval_finish(wealy_eval_plan* p, float* aps, float* r1s, double* sums, void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  if (!p || !aps || !r1s || !sums) return fail(WEALY_ERR_BAD_ARG, "null pointer");
  CU_TRY(cudaMemsetAsync(sums, 0, 3 * sizeof(double), s));
  const int threads = 256;
  const unsigned blocks = (unsigned)ceil_div(p->nq * 32, threads);
  if (p->last_sym) ap_reduce_kernel<<<blocks, threads, 0, s>>>(p->hist, p->s_off, p->cnt, (int)p->nq, aps, r1s, sums, p->sorted_idx);
  else ap_reduce_kernel<<<blocks, threads, 0, s>>>(p->hist, p->off, p->cnt, (int)p->nq, aps, r1s, sums);
  CU_TRY(cudaGetLastError());
  return WEALY_OK;
}

// Per-item ranks of the last run (all ranks' counters summed first in a sharded run): offsets [nq + 1] int64 = CSR
// over the caller's queries, ranks / sims [total_pairs] = every query's relevant items, best first.
extern "C" int wealy_eval_plan_ranks(const wealy_eval_plan* p, int64_t* offsets, int32_t* ranks, float* sims, void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  if (!p || !offsets || !ranks || !sims) return fail(WEALY_ERR_BAD_ARG, "null pointer");
  if (!p->timed) return fail(WEALY_ERR_BAD_ARG, "the plan has not been run yet");
  CU_TRY(cudaMemcpyAsync(offsets, p->off, ((size_t)p->nq + 1) * 8, cudaMemcpyDeviceToDevice, s));
  const int threads = 256;
  const unsigned blocks = (unsigned)ceil_div(p->nq * 32, threads);
  if (p->last_sym)
    rank_export_kernel<<<blocks, threads, 0, s>>>(p->hist, p->thr, p->s_off, p->cnt, (int)p->nq, p->off, p->sorted_idx, ranks, sims);
  else
    rank_export_kernel<<<blocks, threads, 0, s>>>(p->hist, p->thr, p->off, p->cnt, (int)p->nq, p->off, nullptr, ranks, sims);
  CU_TRY(cudaGetLastError());
  return WEALY_OK;
}

// ------------------------------------------------------------------------------------------
// a3: masked reductions
// ------------------------------------------------------------------------------------------
template <typename T>
static int launch_masked(const void* x, const unsigned char* mask, int64_t rows, int64_t cols, int op, float fill,
                         float eps, void* out, cudaStream_t s) {
  if (cols <= 2048 || rows >= 4096) {
    const int threads = 256;
    const unsigned blocks = (unsigned)ceil_div(rows * 32, threads);
    masked_reduce_warp_kernel<T><<<blocks, threads, 0, s>>>((const T*)x, mask, rows, cols, op, fill, eps, (T*)out);
  } else {
    masked_reduce_block_kernel<T><<<(unsigned)rows, 1024, 0, s>>>((const T*)x, mask, rows, cols, op, fill, eps, (T*)out);
  }
  CU_TRY(cudaGetLastError());
  return WEALY_OK;
}

extern "C" int wealy_masked_reduce(const void* x, const uint8_t* mask, int64_t rows, int64_t cols, int dtype, int op,
                                   float fill, float eps, void* out, void* stream) {
  if (rows < 0 || cols < 0) return fail(WEALY_ERR_BAD_ARG, "bad shape rows=%lld cols=%lld", (long long)rows, (long long)cols);
  if (rows == 0) return WEALY_OK;
  if (!x || !out) return fail(WEALY_ERR_BAD_ARG, "null pointer");
  if (op < WEALY_MASKED_SUM || op > WEALY_MASKED_MAX) return fail(WEALY_ERR_BAD_ARG, "unknown masked op %d", op);
  if (rows > 2000000000ll) return fail(WEALY_ERR_UNSUPPORTED, "too many rows");
  cudaStream_t s = (cudaStream_t)stream;
  switch (dtype) {
    case WEALY_F32: return launch_masked<float>(x, mask, rows, cols, op, fill, eps, out, s);
    case WEALY_F16: return launch_masked<__half>(x, mask, rows, cols, op, fill, eps, out, s);
    case WEALY_BF16: return launch_masked<__nv_bfloat16>(x, mask, rows, cols, op, fill, eps, out, s);
    case WEALY_F64:
      masked_reduce_f64_kernel<<<(unsigned)ceil_div(rows * 32, 256), 256, 0, s>>>((const double*)x, mask, rows, cols, op, (double)fill,
                                                                                 (double)eps, (double*)out);
      CU_TRY(cudaGetLastError());
      return WEALY_OK;
    default: return fail(WEALY_ERR_BAD_ARG, "unknown element type %d", dtype);
  }
}

template <typename T, typename A>
static int launch_masked_backward(const void* x, const unsigned char* mask, int64_t rows, int64_t cols, int op, int full,
                                  float fill, float eps, const void* g, void* dx, cudaStream_t s) {
  if (cols <= 2048 || rows >= 4096) {
    const int threads = 256;
    const unsigned blocks = (unsigned)ceil_div(rows * 32, threads);
    masked_reduce_backward_warp_kernel<T, A><<<blocks, threads, 0, s>>>((const T*)x, mask, rows, cols, op, full, (A)fill, (A)eps,
                                                                        (const T*)g, (T*)dx);
  } else {
    masked_reduce_backward_block_kernel<T, A><<<(unsigned)rows, 1024, 0, s>>>((const T*)x, mask, rows, cols, op, full, (A)fill,
                                                                              (A)eps, (const T*)g, (T*)dx);
  }
  CU_TRY(cudaGetLastError());
  return WEALY_OK;
}

extern "C" int wealy_masked_reduce_backward(const void* x, const uint8_t* mask, int64_t rows, int64_t cols, int dtype, int op,
                                            float fill, float eps, int full, const void* g, void* dx, void* stream) {
  if (rows < 0 || cols < 0) return fail(WEALY_ERR_BAD_ARG, "bad shape rows=%lld cols=%lld", (long long)rows, (long long)cols);
  if (rows == 0 || cols == 0) return WEALY_OK;
  if (!x || !g || !dx) return fail(WEALY_ERR_BAD_ARG, "null pointer");
  if (op < WEALY_MASKED_SUM || op > WEALY_MASKED_MAX) return fail(WEALY_ERR_BAD_ARG, "unknown masked op %d", op);
  if (rows > 2000000000ll) return fail(WEALY_ERR_UNSUPPORTED, "too many rows");
  cudaStream_t s = (cudaStream_t)stream;
  switch (dtype) {
    case WEALY_F32: return launch_masked_backward<float, float>(x, mask, rows, cols, op, full, fill, eps, g, dx, s);
    case WEALY_F16: return launch_masked_backward<__half, float>(x, mask, rows, cols, op, full, fill, eps, g, dx, s);
    case WEALY_BF16: return launch_masked_backward<__nv_bfloat16, float>(x, mask, rows, cols, op, full, fill, eps, g, dx, s);
    case WEALY_F64: return launch_masked_backward<double, double>(x, mask, rows, cols, op, full, fill, eps, g, dx, s);
    default: return fail(WEALY_ERR_BAD_ARG, "unknown element type %d", dtype);
  }
}

// a4: distance_tensor_redux (lib/tensor_ops.py:288-373) in one launch -- csrc/redux_kernels.cuh
extern "C" int wealy_distance_redux(const void* dist, const uint8_t* mask, int64_t pairs, int s1, int s2, int dtype, int op,
                                    int karg, int symmetric, float eps, float inf, void* out, void* stream) {
  if (pairs < 0 || s1 < 1 || s2 < 1) return fail(WEALY_ERR_BAD_ARG, "bad shape pairs=%lld s1=%d s2=%d", (long long)pairs, s1, s2);
  if (s1 > kReduxMaxS || s2 > kReduxMaxS) return fail(WEALY_ERR_UNSUPPORTED, "more than %d chunks per track", kReduxMaxS);
  if (op < WEALY_RDX_MIN || op > WEALY_RDX_BPWR) return fail(WEALY_ERR_BAD_ARG, "unknown redux op %d", op);
  if (pairs == 0) return WEALY_OK;
  if (!dist || !out) return fail(WEALY_ERR_BAD_ARG, "null pointer");
  if (pairs > 4ll * 2000000000ll) return fail(WEALY_ERR_UNSUPPORTED, "too many pairs");
  cudaStream_t s = (cudaStream_t)stream;
#define WEALY_RDX(T, A) \
  redux_pairs_kernel<T, A><<<(unsigned)ceil_div(pairs, redux_warps<A>()), 32 * redux_warps<A>(), 0, s>>>((const T*)dist, mask, (long long)pairs, s1, s2, op, karg, symmetric, (A)eps, (A)inf, (T*)out)
  switch (dtype) {
    case WEALY_F32: WEALY_RDX(float, float); break;
    case WEALY_F16: WEALY_RDX(__half, float); break;
    case WEALY_BF16: WEALY_RDX(__nv_bfloat16, float); break;
    case WEALY_F64: WEALY_RDX(double, double); break;
    default: return fail(WEALY_ERR_BAD_ARG, "unknown element type %d", dtype);
  }
#undef WEALY_RDX
  CU_TRY(cudaGetLastError());
  return WEALY_OK;
}

extern "C" int wealy_distance_redux_backward(const void* dist, const uint8_t* mask, int64_t pairs, int s1, int s2, int dtype, int op,
                                             int karg, int symmetric, float eps, float inf, const void* g, void* ddist, void* stream) {
  if (pairs < 0 || s1 < 1 || s2 < 1) return fail(WEALY_ERR_BAD_ARG, "bad shape pairs=%lld s1=%d s2=%d", (long long)pairs, s1, s2);
  if (s1 > kReduxMaxS || s2 > kReduxMaxS) return fail(WEALY_ERR_UNSUPPORTED, "more than %d chunks per track", kReduxMaxS);
  if (op < WEALY_RDX_MIN || op > WEALY_RDX_BPWR) return fail(WEALY_ERR_BAD_ARG, "unknown redux op %d", op);
  if (pairs == 0) return WEALY_OK;
  if (!dist || !g || !ddist) return fail(WEALY_ERR_BAD_ARG, "null pointer");
  if (pairs > 3ll * 2000000000ll) return fail(WEALY_ERR_UNSUPPORTED, "too many pairs");
  cudaStream_t s = (cudaStream_t)stream;
#define WEALY_RDX_BWD(T, A)                                                                                                          \
  redux_pairs_backward_kernel<T, A><<<(unsigned)ceil_div(pairs, redux_bwd_warps<A>()), 32 * redux_bwd_warps<A>(), 0, s>>>(          \
      (const T*)dist, mask, (long long)pairs, s1, s2, op, karg, symmetric, (A)eps, (A)inf, (const T*)g, (T*)ddist)
  switch (dtype) {
    case WEALY_F32: WEALY_RDX_BWD(float, float); break;
    case WEALY_F16: WEALY_RDX_BWD(__half, float); break;
    case WEALY_BF16: WEALY_RDX_BWD(__nv_bfloat16, float); break;
    case WEALY_F64:
      if (pairs > 2000000000ll) return fail(WEALY_ERR_UNSUPPORTED, "too many pairs");
      WEALY_RDX_BWD(double, double);
      break;
    default: return fail(WEALY_ERR_BAD_ARG, "unknown element type %d", dtype);
  }
#undef WEALY_RDX_BWD
  CU_TRY(cudaGetLastError());
  return WEALY_OK;
}

// ------------------------------------------------------------------------------------------
// f3 / f4: the steps either side of the path
// ------------------------------------------------------------------------------------------
template <typename T>
static int launch_mean_pool(const void* x, const uint8_t* mask, int64_t b, int64_t c, int64_t t, void* out, int backward,
                            cudaStream_t s) {
  const long long rows = b * c;
  const int threads = 256;
  const unsigned blocks = (unsigned)ceil_div(rows * 32, threads);
  if (backward)
    mean_pool_bwd_kernel<T><<<blocks, threads, 0, s>>>((const T*)x, mask, rows, (int)c, (int)t, (T*)out);
  else
    mean_pool_fwd_kernel<T><<<blocks, threads, 0, s>>>((const T*)x, mask, rows, (int)c, (int)t, (T*)out);
  CU_TRY(cudaGetLastError());
  return WEALY_OK;
}

extern "C" int wealy_mean_pool(const void* x, const uint8_t* mask, int64_t b, int64_t c, int64_t t, int dtype, void* out,
                               int backward, void* stream) {
  if (b < 0 || c < 0 || t <= 0) return fail(WEALY_ERR_BAD_ARG, "bad shape (%lld, %lld, %lld)", (long long)b, (long long)c, (long long)t);
  if (b * c == 0) return WEALY_OK;
  if (!x || !out) return fail(WEALY_ERR_BAD_ARG, "null pointer");
  if (b * c > 60000000ll || t > 2000000000ll) return fail(WEALY_ERR_UNSUPPORTED, "too large");
  cudaStream_t s = (cudaStream_t)stream;
  switch (dtype) {
    case WEALY_F32: return launch_mean_pool<float>(x, mask, b, c, t, out, backward, s);
    case WEALY_F16: return launch_mean_pool<__half>(x, mask, b, c, t, out, backward, s);
    case WEALY_BF16: return launch_mean_pool<__nv_bfloat16>(x, mask, b, c, t, out, backward, s);
    default: return fail(WEALY_ERR_BAD_ARG, "unknown element type %d", dtype);
  }
}

extern "C" int wealy_segment_mean(const void* x, const int64_t* offsets, int64_t tracks, int64_t dim, int dtype,
                                  float* out, void* stream) {
  if (tracks < 0 || dim <= 0) return fail(WEALY_ERR_BAD_ARG, "bad shape tracks=%lld dim=%lld", (long long)tracks, (long long)dim);
  if (tracks == 0) return WEALY_OK;
  if (!x || !offsets || !out) return fail(WEALY_ERR_BAD_ARG, "null pointer");
  if (tracks > 2000000000ll || dim > 2000000000ll) return fail(WEALY_ERR_UNSUPPORTED, "too large");
  cudaStream_t s = (cudaStream_t)stream;
  const unsigned blocks = (unsigned)tracks;
  switch (dtype) {
    case WEALY_F32: segment_mean_kernel<float><<<blocks, 256, 0, s>>>((const float*)x, (const long long*)offsets, (int)tracks, (int)dim, out); break;
    case WEALY_F16: segment_mean_kernel<__half><<<blocks, 256, 0, s>>>((const __half*)x, (const long long*)offsets, (int)tracks, (int)dim, out); break;
    case WEALY_BF16: segment_mean_kernel<__nv_bfloat16><<<blocks, 256, 0, s>>>((const __nv_bfloat16*)x, (const long long*)offsets, (int)tracks, (int)dim, out); break;
    default: return fail(WEALY_ERR_BAD_ARG, "unknown element type %d", dtype);
  }
  CU_TRY(cudaGetLastError());
  return WEALY_OK;
}

extern "C" int wealy_triplet_mine(const int64_t* z_label, const int64_t* z_idx, int64_t b, int64_t* positives,
                                  int64_t* negatives, void* stream) {
  if (b < 0) return fail(WEALY_ERR_BAD_ARG, "bad batch size");
  if (b == 0) return WEALY_OK;
  if (!z_label || !z_idx || !positives || !negatives) return fail(WEALY_ERR_BAD_ARG, "null pointer");
  if (b > 60000000ll) return fail(WEALY_ERR_UNSUPPORTED, "batch too large");
  const int threads = 256;
  triplet_mine_kernel<<<(unsigned)ceil_div(b * 32, threads), threads, 0, (cudaStream_t)stream>>>(
      (const long long*)z_label, (const long long*)z_idx, (int)b, (long long*)positives, (long long*)negatives);
  CU_TRY(cudaGetLastError());
  return WEALY_OK;
}

template <typename T>
static void launch_triplet_fwd(const void* z, int64_t ldz, int64_t b, int64_t d, const int64_t* pos, const int64_t* neg,
                               float margin, float p, float eps, int swap, float* rows, double* acc, cudaStream_t s) {
  triplet_fwd_kernel<T><<<(unsigned)ceil_div(b * 32, 256), 256, 0, s>>>((const T*)z, ldz, (int)b, (int)d, (const long long*)pos,
                                                                      (const long long*)neg, margin, p, eps, swap,
                                                                      (TripletRow*)rows, acc);
}

extern "C" int wealy_triplet_forward(const void* z, int64_t ldz, int64_t b, int64_t d, int dtype, const int64_t* positives,
                                     const int64_t* negatives, float margin, float p, float eps, int swap, float* rows,
                                     double* acc, void* stream) {
  if (b < 0 || d <= 0 || !(p > 0.f)) return fail(WEALY_ERR_BAD_ARG, "bad shape / norm degree");
  if (!acc) return fail(WEALY_ERR_BAD_ARG, "null pointer");
  cudaStream_t s = (cudaStream_t)stream;
  CU_TRY(cudaMemsetAsync(acc, 0, 2 * sizeof(double), s));
  if (b == 0) return WEALY_OK;
  if (!z || !positives || !negatives || !rows) return fail(WEALY_ERR_BAD_ARG, "null pointer");
  if (b > 60000000ll || d > 2000000000ll) return fail(WEALY_ERR_UNSUPPORTED, "too large");
  switch (dtype) {
    case WEALY_F32: launch_triplet_fwd<float>(z, ldz, b, d, positives, negatives, margin, p, eps, swap, rows, acc, s); break;
    case WEALY_F16: launch_triplet_fwd<__half>(z, ldz, b, d, positives, negatives, margin, p, eps, swap, rows, acc, s); break;
    case WEALY_BF16: launch_triplet_fwd<__nv_bfloat16>(z, ldz, b, d, positives, negatives, margin, p, eps, swap, rows, acc, s); break;
    default: return fail(WEALY_ERR_BAD_ARG, "unknown element type %d", dtype);
  }
  CU_TRY(cudaGetLastError());
  return WEALY_OK;
}

template <typename T>
static void launch_triplet_bwd(const void* z, int64_t ldz, int64_t b, int64_t d, const int64_t* pos, const int64_t* neg,
                               float p, float eps, int swap, const float* rows, const float* upstream, int per_anchor,
                               int mean, const double* acc, float* dz, cudaStream_t s) {
  triplet_bwd_kernel<T><<<(unsigned)ceil_div(b * 32, 256), 256, 0, s>>>((const T*)z, ldz, (int)b, (int)d, (const long long*)pos,
                                                                      (const long long*)neg, p, eps, swap,
                                                                      (const TripletRow*)rows, upstream, per_anchor, mean, acc, dz);
}

extern "C" int wealy_triplet_backward(const void* z, int64_t ldz, int64_t b, int64_t d, int dtype, const int64_t* positives,
                                      const int64_t* negatives, float p, float eps, int swap, const float* rows,
                                      const float* upstream, int per_anchor, int mean, const double* acc, float* dz,
                                      void* stream) {
  if (b < 0 || d <= 0 || !(p > 0.f)) return fail(WEALY_ERR_BAD_ARG, "bad shape / norm degree");
  if (b == 0) return WEALY_OK;
  if (!z || !positives || !negatives || !rows || !upstream || !acc || !dz) return fail(WEALY_ERR_BAD_ARG, "null pointer");
  if (b > 60000000ll || d > 2000000000ll) return fail(WEALY_ERR_UNSUPPORTED, "too large");
  cudaStream_t s = (cudaStream_t)stream;
  CU_TRY(cudaMemsetAsync(dz, 0, (size_t)b * d * sizeof(float), s));
  switch (dtype) {
    case WEALY_F32: launch_triplet_bwd<float>(z, ldz, b, d, positives, negatives, p, eps, swap, rows, upstream, per_anchor, mean, acc, dz, s); break;
    case WEALY_F16: launch_triplet_bwd<__half>(z, ldz, b, d, positives, negatives, p, eps, swap, rows, upstream, per_anchor, mean, acc, dz, s); break;
    case WEALY_BF16: launch_triplet_bwd<__nv_bfloat16>(z, ldz, b, d, positives, negatives, p, eps, swap, rows, upstream, per_anchor, mean, acc, dz, s); break;
    default: return fail(WEALY_ERR_BAD_ARG, "unknown element type %d", dtype);
  }
  CU_TRY(cudaGetLastError());
  return WEALY_OK;
}

#include "loss_api.inl"
