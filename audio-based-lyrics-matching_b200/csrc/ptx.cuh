// Thin inline-PTX wrappers for the sm_100a features the kernels use: mbarrier, TMA
// (cp.async.bulk.tensor), tcgen05 (alloc / mma / commit / ld / fences) and cluster helpers.
// Everything here is __device__ __forceinline__; no CUTLASS / CuTe dependency.
#pragma once
#include <cstdint>
#include <cuda.h>
#include <cuda_runtime.h>

namespace wealy {
namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ uint32_t lane_id() {
  uint32_t l;
  asm volatile("mov.u32 %0, %%laneid;" : "=r"(l));
  return l;
}

// ------------------------------------------------------------------ mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}

__device__ __forceinline__ void fence_mbar_init() {
  // make barrier initialisation visible to the async proxy (TMA / tcgen05.commit)
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// Waiting warps burn issue slots and power that the tensor pipe could use (the sweeps run at the power cap): the
// poll carries a suspend-time hint (the hardware parks the thread until the phase completes or the hint expires) and
// a waiting WARP polls with one lane only (mbar_wait_warp).  Measured on the MMA-bound symmetric sweep: 1-2 %.
constexpr uint32_t kWaitHintNs = 1000;

__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred P;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2, %3;\n"
      "selp.u32 %0, 1, 0, P;\n"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity), "r"(kWaitHintNs)
      : "memory");
  return ok != 0;
}

#ifndef WEALY_DEADLOCK_CYCLES
#define WEALY_DEADLOCK_CYCLES (4000000000ll)  // ~2 s at 2 GHz: a stuck pipeline traps instead of hanging the GPU
#endif

// The deadlock clock of a waiting thread: read once per kClockPolls failed polls, not per poll (the poll loops are a
// fifth of the symmetric sweep's executed instructions).  The first read starts the count, so a wait that ends within
// kClockPolls polls reads no clock at all; a stuck protocol still traps within seconds.
constexpr int kClockPolls = 2048;
struct DeadlockClock {
  long long t0 = 0;
  int polls = 0;
  __device__ __forceinline__ void tick(const char* what, uint64_t* bar, uint32_t parity) {
    if (++polls < kClockPolls) return;
    polls = 0;
    const long long now = clock64();
    if (t0 == 0) {
      t0 = now;
    } else if (now - t0 > WEALY_DEADLOCK_CYCLES) {
      printf("wealy: %s deadlock block=%d thread=%d bar=0x%x parity=%u\n", what, (int)blockIdx.x, (int)threadIdx.x,
             smem_u32(bar), parity);
      __trap();
    }
  }
};

// Spin on the barrier phase.  try_wait suspends in hardware for a bounded time; the clock check turns a protocol bug
// into a trap (reported as a CUDA error) instead of a hang that would take the whole GPU box down.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  DeadlockClock clk;
  while (!mbar_try_wait(bar, parity)) clk.tick("mbarrier", bar, parity);
}

// The same for a whole warp: one lane polls, the others wait at the warp barrier (32x fewer polling lanes)
__device__ __forceinline__ void mbar_wait_warp(uint64_t* bar, uint32_t parity) {
  if (lane_id() == 0) mbar_wait(bar, parity);
  __syncwarp();
}

// barrier among a subset of the CTA's warps (id 0 is __syncthreads)
__device__ __forceinline__ void named_barrier_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// ------------------------------------------------------------------ TMA
__device__ __forceinline__ void prefetch_tensormap(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}

// 2-D tiled load global -> shared, completion counted in bytes on `bar`.  c0 = innermost coord.
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int32_t c0,
                                            int32_t c1, uint64_t cache_policy) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4}], [%2], %5;"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1),
        "l"(cache_policy)
      : "memory");
}

// 1-D bulk copy global -> shared (16-byte aligned, size a multiple of 16), completion counted in bytes on `bar`
__device__ __forceinline__ void bulk_load(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(gsrc)), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}

// L2 eviction-priority policies (createpolicy encodings used by cp.async.bulk cache hints)
constexpr uint64_t kEvictNormal = 0x1000000000000000ull;
constexpr uint64_t kEvictFirst = 0x12F0000000000000ull;
constexpr uint64_t kEvictLast = 0x14F0000000000000ull;

// ------------------------------------------------------------------ tcgen05 / TMEM
template <uint32_t kCols>
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result) {
  static_assert(kCols >= 32 && kCols <= 512 && (kCols & (kCols - 1)) == 0, "TMEM columns: power of two in [32,512]");
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)),
               "n"(kCols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}

template <uint32_t kCols>
__device__ __forceinline__ void tmem_dealloc(uint32_t tmem_addr) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_addr), "n"(kCols) : "memory");
}

__device__ __forceinline__ void tc_fence_before_sync() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after_sync() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

// D[tmem] (+)= A[smem] * B[smem]; kind::f16 covers fp16 and bf16 inputs with fp32 accumulation.
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                         uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}

// Arrive on `bar` once every tcgen05.mma issued so far by this thread has completed
// (implies tcgen05.fence::before_thread_sync).
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// TMEM -> registers: this warp's 32 lanes (one accumulator row per thread) x 32 consecutive
// fp32 columns starting at `taddr` (lane field = first lane of the warp's quadrant).
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}

__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }


// ------------------------------------------------------------------ CTA pairs (clusters of two, cta_group::2)
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t cluster_id_x() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%clusterid.x;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t n_clusters_x() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%nclusterid.x;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of `p` (a shared-memory object of THIS CTA) as seen in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t map_to_cta(const void* p, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_u32(p)), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// The same without release semantics: for hand-overs that publish nothing through memory (an epilogue warp telling the
// MMA thread that it has read its accumulator chunk: the tcgen05.ld data already sits in registers).  The release
// form compiles to MEMBAR.ALL.GPU + ERRBAR and waits for every outstanding global RED of the warp -- measured as
// 12 % of all stall samples of the pair kernel.
__device__ __forceinline__ void mbar_arrive_cluster_relaxed(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void st_cluster_u32(uint32_t cluster_addr, uint32_t v) {
  asm volatile("st.shared::cluster.u32 [%0], %1;" ::"r"(cluster_addr), "r"(v) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait_cluster(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  // (with the suspend-time hint of mbar_try_wait: an un-hinted poll loop was 25 % of the pair kernel's instructions)
  asm volatile(
      "{\n"
      ".reg .pred P;\n"
      "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 P, [%1], %2, %3;\n"
      "selp.u32 %0, 1, 0, P;\n"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity), "r"(kWaitHintNs)
      : "memory");
  return ok != 0;
}

// wait with cluster-scope acquire: the barrier is signalled by the peer CTA
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait_cluster(bar, parity)) return;
  DeadlockClock clk;
  while (!mbar_try_wait_cluster(bar, parity)) clk.tick("cluster mbarrier", bar, parity);
}

// a whole warp waiting on a cluster-scope barrier: one lane polls (see mbar_wait_warp)
__device__ __forceinline__ void mbar_wait_cluster_warp(uint64_t* bar, uint32_t parity) {
  if (lane_id() == 0) mbar_wait_cluster(bar, parity);
  __syncwarp();
}

// 2-D tiled load issued by either CTA of a pair; completion bytes are counted on the barrier at `leader_bar_addr`
// (a shared::cluster address inside the LEADER CTA, rank 0 of the pair)
__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const CUtensorMap* m, uint32_t leader_bar_addr, int32_t c0,
                                                 int32_t c1, uint64_t cache_policy) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4}], [%2], %5;"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(leader_bar_addr), "r"(c0), "r"(c1),
        "l"(cache_policy)
      : "memory");
}

template <uint32_t kCols>
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* smem_result) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)), "n"(kCols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <uint32_t kCols>
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t tmem_addr) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_addr), "n"(kCols) : "memory");
}

// D[tmem of both CTAs] (+)= A[smem of each CTA: its 128 rows] * B[smem: each CTA holds half of the N columns]
__device__ __forceinline__ void umma_f16_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                              uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on the barrier at the same shared-memory offset in BOTH CTAs once the MMAs issued so far have completed
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
      ::"r"(smem_u32(bar)), "h"((uint16_t)3)
      : "memory");
}

// ------------------------------------------------------------------ descriptors
// Shared-memory matrix descriptor for a K-major operand tile written by TMA with the given
// swizzle (row pitch == swizzle span).  Field layout (PTX ISA "tcgen05 shared memory descriptor"):
//   [0,14)  start address >> 4          [16,30) leading-dim byte offset >> 4 (unused for swizzled K-major; 1)
//   [32,46) stride-dim byte offset >> 4 (distance between 8-row groups)   [46,48) version = 1
//   [61,64) layout: 0 none, 2 = 128B swizzle, 4 = 64B swizzle, 6 = 32B swizzle
template <int kSwizzleBytes>
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr) {
  static_assert(kSwizzleBytes == 128 || kSwizzleBytes == 64 || kSwizzleBytes == 32, "swizzle span");
  constexpr uint64_t layout = kSwizzleBytes == 128 ? 2ull : (kSwizzleBytes == 64 ? 4ull : 6ull);
  constexpr uint64_t sbo = (8ull * kSwizzleBytes) >> 4;  // 8 rows of one swizzle span each
  return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | (1ull << 16) | (sbo << 32) | (1ull << 46) | (layout << 61);
}

// Instruction descriptor for tcgen05.mma kind::f16, fp32 accumulate, both operands K-major.
//   [4,6) D format (1 = f32)  [7,10) A format  [10,13) B format (0 = f16, 1 = bf16)
//   [15] A major  [16] B major (0 = K)  [17,23) N >> 3  [24,29) M >> 4
__host__ __device__ constexpr uint32_t make_idesc_f16(int m, int n, bool bf16) {
  return (1u << 4) | ((bf16 ? 1u : 0u) << 7) | ((bf16 ? 1u : 0u) << 10) | ((uint32_t)(n >> 3) << 17) |
         ((uint32_t)(m >> 4) << 24);
}

}  // namespace ptx
}  // namespace wealy
