// tcgen05_utils.cuh -- PTX wrappers shared by the tensor-core kernels (scan_mma.cu, selfjoin_mma.cu):
// mbarrier, TMA bulk tensor loads, tcgen05 MMA / commit / TMEM loads, the K-major SWIZZLE_128B
// shared-memory descriptor and the kind::f16 instruction descriptor (layouts as documented for
// sm_100 in the CUTLASS headers cute/arch/mma_sm100_desc.hpp), plus the host-side tensor-map builder.
#pragma once
#include <cuda.h>

#include "common.cuh"

namespace mmrs {

constexpr uint32_t kWatchdogSpins = 1u << 24;

// ---- PTX wrappers ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a pipeline bug must end the kernel with a status flag, not hang the GPU.
__device__ __forceinline__ bool mbar_wait(uint64_t* bar, uint32_t parity, volatile uint32_t* abort_flag, int32_t* flags) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (*abort_flag) return false;
    if (++spins > kWatchdogSpins) {
      *abort_flag = 1;
      atomicOr(flags, kFlagWatchdog);
      return false;
    }
  }
  return true;
}
// one lane of a converged warp
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, uint64_t* bar,
                                            int32_t c0, int32_t c1, uint64_t cache_hint) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4}], [%2], %5;"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0),
      "r"(c1), "l"(cache_hint)
      : "memory");
}
// request a tile into L2 only (no shared-memory destination, no barrier)
__device__ __forceinline__ void tma_prefetch_2d(const CUtensorMap* map, int32_t c0, int32_t c1) {
  asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global [%0, {%1, %2}];"
               ::"l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tcgen05_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// kind::i8: signed int8 A / B, s32 accumulator, K = 32 per instruction
__device__ __forceinline__ void umma_i8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                        uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// 32 lanes x 16 consecutive fp32 columns: thread i of the warp gets TMEM lane (base + i)
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---- CTA pair (cta_group::2): two SMs of one TPC run ONE MMA of M = 256 -----------------------
// Each CTA stages its own 128 rows of A and HALF of B's rows; the tensor cores of both SMs read
// the two B halves over the pair link, so per SM the TMA fill and the shared-memory operand reads
// drop from A + B to A + B/2 per MMA (L2 -> SM bytes of a C5-shaped scan: 35.8 -> 23.9 GB, ring
// stages 48 -> 32 KB; profiles/r01_k2_c5like*_summary.txt, same-box A/B in profiles/r01_pair_ab.log).
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
// shared::cluster address of the same variable in CTA `rank` of this cluster
__device__ __forceinline__ uint32_t mapa_u32(uint32_t smem_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// Arrive on a barrier of another CTA of the cluster.  Default (CTA-scope) release semantics on
// purpose: `.release.cluster` compiles to a cluster-wide ERRBAR that waits for every global store
// and atomic the warp still has in flight -- 17 % of all warp samples of the pair kernel's
// epilogue (profiles/r01_k2_c5like_pair_summary.txt).  What the arrival publishes here are
// finished TMEM reads, which tcgen05.fence::before_thread_sync orders.
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// TMA load into THIS CTA's shared memory whose byte count is credited to a barrier that may live
// in the peer CTA (the pair leader's `full` barrier collects both halves of a stage)
__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const CUtensorMap* map, uint32_t bar_cluster_addr,
                                                 int32_t c0, int32_t c1, uint64_t cache_hint) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4}], [%2], %5;"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar_cluster_addr), "r"(c0),
      "r"(c1), "l"(cache_hint)
      : "memory");
}
__device__ __forceinline__ void umma_bf16_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_i8_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::i8 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrives (once the MMAs issued so far retire) on the barrier at this offset in BOTH CTAs of the pair
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
      ::"r"(smem_u32(bar)), "h"(static_cast<uint16_t>(3))
      : "memory");
}

// K-major SWIZZLE_128B shared-memory matrix descriptor (sm_100 "version 1"): rows are 128 bytes,
// 8-row core groups are 1024 bytes apart (SBO); LBO is unused for swizzled K-major layouts.
__device__ __forceinline__ uint64_t make_sw128_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3ffffu) >> 4);       // start address, bits [0,14)
  d |= static_cast<uint64_t>(1) << 16;                           // leading byte offset (>>4), unused
  d |= static_cast<uint64_t>(1024 >> 4) << 32;                   // stride byte offset (>>4)
  d |= static_cast<uint64_t>(1) << 46;                           // descriptor version (Blackwell)
  d |= static_cast<uint64_t>(2) << 61;                           // layout type: SWIZZLE_128B
  return d;
}
// kind::f16 instruction descriptor: D fp32, A/B bf16, both K-major, M=128, N=n.
__host__ __device__ constexpr uint32_t make_idesc(uint32_t n, uint32_t m = 128u) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((n >> 3) << 17) | ((m >> 4) << 24);
}
// kind::i8 instruction descriptor: D s32 (c_format 2), A/B signed int8 (format 1), both K-major, M=128, N=n.
__host__ __device__ constexpr uint32_t make_idesc_i8(uint32_t n, uint32_t m = 128u) {
  return (2u << 4) | (1u << 7) | (1u << 10) | ((n >> 3) << 17) | ((m >> 4) << 24);
}

constexpr uint64_t kEvictFirst = 0x12F0000000000000ull;   // gallery: streamed once
constexpr uint64_t kEvictLast = 0x14F0000000000000ull;    // queries: re-read by every tile
constexpr uint64_t kEvictNormal = 0x1000000000000000ull;  // gallery tile that the same SM pair re-reads for the next query chunk

// ---- host side ---------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);

inline EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// 2-D bf16 row-major [rows, cols] tensor with row stride ld (elements); box = [box_rows, 64 cols]
inline bool make_map(CUtensorMap* map, const void* base, uint64_t rows, uint64_t cols, uint64_t ld,
                     uint32_t box_rows) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return false;
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {ld * 2};
  cuuint32_t box[2] = {64u, box_rows};
  cuuint32_t estr[2] = {1, 1};
  return fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

}  // namespace mmrs
