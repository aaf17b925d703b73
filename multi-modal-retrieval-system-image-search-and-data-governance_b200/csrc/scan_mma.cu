// scan_mma.cu -- K2: tcgen05 tensor-core scan for batched queries over a bf16 (or int8, kind::i8) gallery.
//
// "Batched queries really are a dense contraction" (BASELINE.json): scores[128 rows, Q] =
// G_tile[128, D] * Qmat[Q, D]^T, both operands K-major bf16.  One persistent CTA per SM walks its
// share of the 128-row gallery tiles:
//
//   warp 0 (one lane)  TMA producer: per 64-column k-block one 128x64 gallery box (HBM stream)
//                      and one Qx64 query box (L2 resident) into a SWIZZLE_128B smem ring
//   warp 1 (one lane)  tcgen05.mma issuer: D[tmem] (+)= A[smem] * B[smem], M=128, N=Q, K=16;
//                      tcgen05.commit frees the smem slot / publishes the accumulator
//   warp 2             TMEM allocator (2 accumulator stages of Q fp32 columns)
//   warps 4..11        epilogue: tcgen05.ld the 128xQ accumulator (one gallery row per thread,
//                      two warps per TMEM lane quarter splitting the columns)
//                      and run the same three epilogues as K1 -- the score matrix never reaches
//                      HBM unless kModeScores asks for it.
//
// The accumulator is double buffered so the epilogue of tile i overlaps the MMAs of tile i+1.
// Roofline: HBM-bound (N*D*2 bytes per pass) up to Q ~ 200, tensor-bound beyond
// (SURVEY.md section 8d).
//
// PAIR mode (more than 64 queries): the grid is launched as clusters of two CTAs (one TPC) that
// run ONE tcgen05.mma.cta_group::2 of M = 256: each CTA stages its own gallery tile (A, 128 rows)
// and HALF of the query chunk (B); CTA 0's MMA warp issues for both, each CTA's accumulator
// (its 128 rows x all queries of the chunk) lands in its own TMEM and is read out by its own
// epilogue warps.  The pair halves the query-operand traffic per SM (TMA fill and shared-memory
// reads: A + B/2 instead of A + B per MMA; L2 -> SM bytes of a C5-shaped scan 35.8 -> 23.9 GB) and
// makes the ring stages 32 instead of 48 KB; same-box A/B: +11-14 % under the power cap
// (profiles/r01_pair_ab.log, profiles/r01_k2_c5like*_summary.txt).  Work units of a
// pair are (tile pair, query chunk) in chunk-minor order, so the chunks of one tile pair are
// scanned by neighbouring pairs at the same time and share the tile through L2.
#include <stdlib.h>

#include "plan.h"
#include "tcgen05_utils.cuh"

namespace mmrs {

constexpr int kCtrlWarps = 4;            // TMA producer, MMA issuer, TMEM allocator, spare
constexpr int kMaxEpiWarps = 16;         // epilogue warps: 8 (two CTAs per SM) or 16 (tensor-bound batches)
constexpr int kBlockM = kTileRows;       // gallery rows per tile == UMMA M
constexpr int kBlockK = 64;              // bf16 elements per k-block == one 128-byte swizzle row
constexpr int kUmmaK = 16;
constexpr int kMaxQ = 256;               // UMMA N limit
constexpr int kSplitMaxQ = 48;           // fp32 emulation, single CTA: queries per pass (3 x (16 + 6) KB per stage, 3 stages)
constexpr int kSplitPairMaxQ = 128;      // fp32 emulation as CTA pairs: each CTA stages half the query rows of every plane
constexpr int kMaxQChunks = 4;           // query chunks of kMaxQ that may share the gallery stream of one launch
constexpr int kABytes = kBlockM * kBlockK * 2;   // 16 KiB
constexpr int kMaxStages = 8;
constexpr uint32_t kStash = 4;            // parked candidates per epilogue thread before a flush

template <int CHUNKS, int EPI = kMaxEpiWarps>   // query chunks whose thresholds a CTA keeps (1, or kMaxQChunks in pair mode); epilogue warps
struct MmaSharedT {
  uint64_t full[kMaxStages];
  uint64_t empty[kMaxStages];
  uint64_t tmem_full[2];
  uint64_t tmem_empty[2];
  uint32_t tmem_base;
  volatile uint32_t abort;
  alignas(16) float thr[kMaxQ * CHUNKS];       // exact bound on the scaled score
  alignas(16) float thr_raw[kMaxQ * CHUNKS];   // conservative bound on the RAW accumulator (thr / scale, nudged down)
  alignas(16) uint2 stash[EPI][kStash * 32];  // per epilogue thread: parked (column, score) pairs
};

// Label-conditioned launches keep their query labels in a tail behind the shared struct, laid out like
// thr (column c of chunk ch at ch * kMaxQ + c); only they size it in, so an unlabeled launch keeps its
// shared-memory footprint and its ring stages.  Slots of the tail:
__host__ __device__ __forceinline__ int label_tail_slots(bool pair, int n_qchunks, int n_umma) {
  return pair && n_qchunks > 1 ? n_qchunks * kMaxQ : n_umma;
}

struct MmaCfg {
  int32_t n_umma;        // UMMA N: queries of this pass rounded up to 16
  int32_t k_blocks;      // ceil(dim / 64)
  int32_t stages;
  int32_t tmem_cols;     // power of two >= 2 * n_umma, >= 32
  int32_t acc_stride;    // column offset between the two accumulator stages
  int32_t split;         // 1: bf16 operands; 3: fp32 emulation, operands split into hi/mid/lo bf16 planes
  int64_t g_plane_rows;  // split == 3: rows between two planes of the gallery (= n_rows)
  int32_t q_plane_rows;  // split == 3: rows between two planes of the prepared queries
  int32_t debug_skip_epilogue;   // measurement aid (MMRS_K2_DEBUG_SKIP_EPI=1): results are garbage
  int32_t n_qchunks;     // pair mode: query chunks of kMaxQ in this launch (they are work units, not gridDim.y)
  int32_t sticky;        // pair mode, several chunks, many tiles: a pair scans ALL chunks of its tile pair back to back
  int32_t prefetch;      // TMA-prefetch the gallery tile of the NEXT unit into L2 while this unit's tile is loaded
};



// SPLIT is a template parameter on purpose: with the operand-plane count a run-time value the single lane that
// issues tcgen05.mma carried both code paths and the C5-shaped scan fell from 4.11 back to 4.67 ms per launch
// (profiles/r02_prefetch_ab.log against r02_sticky_ab.log) -- that loop is issue-bound, every instruction counts.
// LABELED: label-conditioned search (p.row_labels != nullptr, dense / filter modes only), a separate
// instantiation so that the unlabeled kernels keep their code and registers.
// I8: int8 gallery and query rows (include/mmrs_b200.h, "int8 galleries").  The TMA boxes move the same
// 128-byte rows (128 codes per k-block), tcgen05.mma.kind::i8 takes K = 32 per instruction -- four per
// k-block, the same +32-byte descriptor step -- into an s32 accumulator, and the epilogue turns each exact
// int32 sum into i8_score with a_q from shared memory (the thr_raw slots, unused by int8) and the row's scale
// s_r from the row's tail.  Every pair's exact score is compared with thr: no raw-accumulator prefilter.
template <int MODE, int EPI_WARPS, bool PAIR, int SPLIT, bool LABELED = false, bool I8 = false>
__global__ void __launch_bounds__((kCtrlWarps + EPI_WARPS) * 32, EPI_WARPS == 8 ? 2 : 1)
scan_mma_kernel(const __grid_constant__ CUtensorMap map_g, const __grid_constant__ CUtensorMap map_q,
                const ScanParams p, const MmaCfg cfg, int32_t* flags) {
  // the two-per-SM variants (8 epilogue warps) scan ONE query chunk and keep the small layout
  using Shared = MmaSharedT<(PAIR && EPI_WARPS == 16) ? kMaxQChunks : 1, EPI_WARPS>;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // dynamic smem: [stages x (A 16 KiB | B rows*128 B)] then Shared; the ring must be
  // 1024-byte aligned for the 128-byte swizzle.  B rows: n_umma, in pair mode n_umma / 2.
  uint8_t* ring = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int b_rows = PAIR ? cfg.n_umma / 2 : cfg.n_umma;
  const uint32_t b_bytes = static_cast<uint32_t>(b_rows) * kBlockK * 2;
  // split == 3 (fp32 emulation): a stage holds the hi/mid/lo planes of both operands,
  // [A_hi | A_mid | A_lo | B_hi | B_mid | B_lo]
  const uint32_t a_all = static_cast<uint32_t>(SPLIT) * kABytes;
  const uint32_t stage_bytes = static_cast<uint32_t>(SPLIT) * (kABytes + b_bytes);
  Shared* sh = reinterpret_cast<Shared*>(ring + static_cast<size_t>(cfg.stages) * stage_bytes);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // Warp roles.  The epilogue warps take the LOW warp ids and the three control warps the highest:
  // the warp schedulers favour the higher warp id among ready warps (B300_MICROARCH.md, arbiter:
  // hi-wid-first), so the single threads that issue TMA and tcgen05.mma cannot be queued behind
  // sixteen busy epilogue warps.  (Measured on B200 it made no difference -- 213 vs 211 us at 256
  // queries: the 29 us the read-out costs there is TMEM-port time, not issue slots -- but it is the
  // order that cannot hurt.)  TMEM lane quarters go by warp id % 4, unaffected.
  constexpr int kTmaWarp = EPI_WARPS, kMmaWarp = EPI_WARPS + 1, kAllocWarp = EPI_WARPS + 2;

  // ---- work units ---------------------------------------------------------------------------
  // A unit is one accumulator tile: (gallery tile, query chunk).  Without pairs, CTA (x, y) walks
  // j = x, x + gridDim.x, ... (skipping the tiles an earlier phase covered) for the kMaxQ queries of
  // chunk y: the chunks' CTAs walk the same tile sequence at the same pace, so all but the first
  // find the tile in L2 and the HBM stream per query is divided by gridDim.y.  In pair mode the
  // pair walks units u = pair, pair + n_pairs, ...: u -> (tile pair u / n_qchunks, chunk
  // u % n_qchunks) over the VISITED tiles only; CTA `rank` of the pair takes tile 2 * (tile pair) + rank.
  const int inc = p.sched.tile_inc, exc = p.sched.tile_exc;
  const uint32_t rank = PAIR ? cluster_ctarank() : 0u;
  const int R = PAIR ? plan_exclusion_ratio(inc, exc) : 0;
  const int n_valid = plan_n_visited(p.sched.n_sel, R);
  // Sticky order (several chunks, many tiles -- the tensor-bound 64K-query batches): the pair takes tile
  // pairs tp = pair, pair + n_pairs, ... and scans all n_ch chunks of one tile pair back to back, so the
  // three re-reads of a gallery tile come from L2 BY CONSTRUCTION (the same SM pair asks again a few
  // microseconds later) instead of relying on four different pairs staying in step: the interleaved order
  // read every tile from DRAM about twice (dram read 5.86 GB for 2.98 GB of gallery, L2 hit rate 70 %,
  // profiles/r01_k2_c5like_pair2_summary.txt).
  const int n_ch = PAIR ? cfg.n_qchunks : 1;
  const bool sticky = PAIR && cfg.sticky != 0;
  const int n_pairs_grid = static_cast<int>(gridDim.x >> 1), pair_id = static_cast<int>(blockIdx.x >> 1);
  const int u_begin = PAIR ? (sticky ? 0 : pair_id) : static_cast<int>(blockIdx.x);
  const int u_step = PAIR ? (sticky ? 1 : n_pairs_grid) : static_cast<int>(gridDim.x);
  const int n_tile_pairs = (n_valid + 1) / 2;
  const int n_units = PAIR ? (sticky ? (pair_id < n_tile_pairs ? ((n_tile_pairs - pair_id + n_pairs_grid - 1) / n_pairs_grid) * n_ch : 0)
                                     : plan_pair_units(n_valid, n_ch))
                           : p.sched.n_sel;
  struct Unit { int j, chunk; bool valid, skip; };
  auto unit_of = [&](int u) -> Unit {
    if constexpr (PAIR) {
      // sticky: u counts this pair's own units; u / n_ch-th tile pair of the pair, chunk u % n_ch
      const int gu = sticky ? (pair_id + (u / n_ch) * n_pairs_grid) * n_ch + u % n_ch : u;
      const PairUnit pu = plan_pair_unit(gu, static_cast<int>(rank), n_ch, n_valid, R);   // plan.h
      return Unit{pu.j, pu.chunk, pu.valid, false};
    } else {
      return Unit{u, static_cast<int>(blockIdx.y), true, exc != 0 && ((u * inc) % exc) == 0};
    }
  };

  if (threadIdx.x == 0) {
    for (int s = 0; s < cfg.stages; ++s) { mbar_init(&sh->full[s], 1); mbar_init(&sh->empty[s], 1); }
    // pair mode: the leader's tmem_empty collects the epilogue warps of both CTAs
    for (int a = 0; a < 2; ++a) { mbar_init(&sh->tmem_full[a], 1); mbar_init(&sh->tmem_empty[a], PAIR ? 2 * EPI_WARPS : EPI_WARPS); }
    sh->abort = 0;
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&map_g)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&map_q)) : "memory");
  }
  pdl_launch_dependents();
  if (warp == kAllocWarp) {
    if constexpr (PAIR) {   // both CTAs of the pair, same warp id, same destination offset
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&sh->tmem_base)),
                   "r"(static_cast<uint32_t>(cfg.tmem_cols))
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&sh->tmem_base)),
                   "r"(static_cast<uint32_t>(cfg.tmem_cols))
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  pdl_wait();   // everything above overlaps the predecessor; its results are read from here on
  // The hot loop compares the RAW accumulator with thr / scale (no multiply per score); that bound
  // is nudged down by a few ulps so that it can only let MORE through, and the rare path repeats the
  // exact test `scale * acc >= thr` before parking a candidate.  Non-positive scales keep the
  // multiply (raw_ok = false).
  const bool raw_ok = p.scale > 0.f;
  constexpr bool labeled = LABELED && MODE != kModeScores;
  int32_t* lab_s = reinterpret_cast<int32_t*>(sh + 1);                   // the label tail (labeled launches only)
  {
    const int first_q = PAIR ? p.q0 : p.q0 + static_cast<int>(blockIdx.y) * kMaxQ;
    const int n_q = PAIR ? p.nq : min(p.nq - static_cast<int>(blockIdx.y) * kMaxQ, kMaxQ);
    for (int c = threadIdx.x; c < kMaxQ * (PAIR ? kMaxQChunks : 1); c += (kCtrlWarps + EPI_WARPS) * 32) {
      float t = __int_as_float(0x7f800000);  // +inf: padded columns never pass the filter
      if (MODE == kModeFilter && c < n_q && cfg.debug_skip_epilogue != 2) t = p.thr[first_q + c];
      sh->thr[c] = t;
      float tr = t;
      if (raw_ok && isfinite(t)) {
        tr = t / p.scale;
        tr = tr - fabsf(tr) * 4.8e-7f - 1e-37f;
      }
      if constexpr (I8)   // a_q = fl(s_q * scale); padded columns 0
        tr = c < n_q ? __fmul_rn(i8_row_scale(reinterpret_cast<const int8_t*>(p.queries) +
                                                  static_cast<size_t>(first_q + c) * p.ldq, p.dim), p.scale)
                     : 0.f;
      sh->thr_raw[c] = tr;
    }
    if constexpr (labeled) {
      const int n_lab = label_tail_slots(PAIR, cfg.n_qchunks, cfg.n_umma);
      for (int c = threadIdx.x; c < n_lab; c += (kCtrlWarps + EPI_WARPS) * 32)
        lab_s[c] = c < n_q ? __ldg(p.query_labels + first_q + c) : -1;   // padded columns never pass anyway
    }
  }
  tcgen05_fence_before();
  if constexpr (PAIR) {
    __syncwarp();
    cluster_sync_all();   // the peer's barriers are initialised before anything is signalled across
  } else {
    __syncthreads();
  }
  tcgen05_fence_after();
  const uint32_t tmem_base = sh->tmem_base;

  if (warp == kTmaWarp) {
    // ===== TMA producer =====
    if (lane == 0) {
      uint32_t stage = 0, phase = 0;
      bool ok = true;
      for (int u = u_begin; u < n_units && ok; u += u_step) {
        const Unit un = unit_of(u);
        if (un.skip) continue;
        const int32_t row0 = un.j * inc * kBlockM;
        const int32_t qrow0 = p.q0 + un.chunk * kMaxQ + static_cast<int>(rank) * b_rows;
        if (cfg.prefetch) {
          // the next unit this CTA will load a NEW gallery tile for (sticky: the chunks of a tile pair re-read it)
          int u2 = u + u_step;
          while (u2 < n_units && unit_of(u2).skip) u2 += u_step;
          if (u2 < n_units) {
            const Unit nx = unit_of(u2);
            if (nx.j != un.j) {
              const int32_t nrow0 = nx.j * inc * kBlockM;
              for (int pl = 0; pl < SPLIT; ++pl)
                for (int kb = 0; kb < cfg.k_blocks; ++kb)
                  tma_prefetch_2d(&map_g, kb * kBlockK, static_cast<int32_t>(pl * cfg.g_plane_rows) + nrow0);
            }
          }
        }
        for (int kb = 0; kb < cfg.k_blocks; ++kb) {
          if (!mbar_wait(&sh->empty[stage], phase ^ 1, &sh->abort, flags)) { ok = false; break; }
          uint8_t* a_dst = ring + static_cast<size_t>(stage) * stage_bytes;
          if constexpr (PAIR) {
            // both halves of the stage are credited to the LEADER's barrier, which its MMA warp waits on
            const uint32_t full_leader = mapa_u32(smem_u32(&sh->full[stage]), 0);
            if (rank == 0) mbar_expect_tx(&sh->full[stage], 2 * stage_bytes);
            const uint64_t a_hint = sticky ? (un.chunk == n_ch - 1 ? kEvictFirst : kEvictNormal) : kEvictFirst;
#pragma unroll
            for (int pl = 0; pl < SPLIT; ++pl) {
              tma_load_2d_pair(a_dst + pl * kABytes, &map_g, full_leader, kb * kBlockK,
                               static_cast<int32_t>(pl * cfg.g_plane_rows) + row0, a_hint);
              tma_load_2d_pair(a_dst + a_all + pl * b_bytes, &map_q, full_leader, kb * kBlockK,
                               pl * cfg.q_plane_rows + qrow0, kEvictLast);
            }
          } else {
            mbar_expect_tx(&sh->full[stage], stage_bytes);
#pragma unroll
            for (int pl = 0; pl < SPLIT; ++pl) {
              tma_load_2d(a_dst + pl * kABytes, &map_g, &sh->full[stage], kb * kBlockK,
                          static_cast<int32_t>(pl * cfg.g_plane_rows) + row0, kEvictFirst);
              tma_load_2d(a_dst + a_all + pl * b_bytes, &map_q, &sh->full[stage], kb * kBlockK,
                          pl * cfg.q_plane_rows + qrow0, kEvictLast);
            }
          }
          if (++stage == static_cast<uint32_t>(cfg.stages)) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == kMmaWarp) {
    // ===== MMA issuer (pair mode: the leader CTA issues for both) =====
    // The WHOLE warp walks the loop and one elected lane issues: with the loop inside `if (lane == 0)`
    // every descriptor lived in vector registers and each tcgen05.mma cost an ELECT + five R2UR +
    // predicate shuffling -- ~125 instructions and 778 clocks per k-block against the 512 clocks its
    // four MMAs keep the tensor pipe busy (ncu: ring always full, pipe 66 % active,
    // profiles/r01_k2_c5like_summary.txt).  Warp-uniform code keeps them in uniform registers.
    if (rank == 0) {
      const uint32_t idesc = I8 ? make_idesc_i8(static_cast<uint32_t>(cfg.n_umma), PAIR ? 256u : 128u)
                                : make_idesc(static_cast<uint32_t>(cfg.n_umma), PAIR ? 256u : 128u);
      const uint32_t ring_addr = smem_u32(ring);
      uint32_t stage = 0, phase = 0, it = 0;
      bool ok = true;
      for (int u = u_begin; u < n_units && ok; u += u_step) {
        if (unit_of(u).skip) continue;
        const uint32_t as = it & 1, aphase = (it >> 1) & 1;
        if (!__all_sync(0xffffffffu, mbar_wait(&sh->tmem_empty[as], aphase ^ 1, &sh->abort, flags))) break;
        tcgen05_fence_after();
        const uint32_t d_tmem = tmem_base + as * static_cast<uint32_t>(cfg.acc_stride);
        for (int kb = 0; kb < cfg.k_blocks; ++kb) {
          if (!__all_sync(0xffffffffu, mbar_wait(&sh->full[stage], phase, &sh->abort, flags))) { ok = false; break; }
          tcgen05_fence_after();
          const uint32_t a_addr = ring_addr + stage * stage_bytes;
          if (elect_one()) {
            if constexpr (I8) {
              const uint64_t adesc = make_sw128_desc(a_addr);
              const uint64_t bdesc = make_sw128_desc(a_addr + kABytes);
#pragma unroll
              for (int k = 0; k < kBlockK / kUmmaK; ++k) {   // 32 codes = 32 bytes per instruction
                if constexpr (PAIR)
                  umma_i8_pair(d_tmem, adesc + static_cast<uint64_t>(k * 2), bdesc + static_cast<uint64_t>(k * 2), idesc,
                               (kb | k) != 0 ? 1u : 0u);
                else
                  umma_i8(d_tmem, adesc + static_cast<uint64_t>(k * 2), bdesc + static_cast<uint64_t>(k * 2), idesc,
                          (kb | k) != 0 ? 1u : 0u);
              }
            } else if constexpr (SPLIT == 1) {
              const uint64_t adesc = make_sw128_desc(a_addr);
              const uint64_t bdesc = make_sw128_desc(a_addr + kABytes);
#pragma unroll
              for (int k = 0; k < kBlockK / kUmmaK; ++k) {
                // advancing 16 bf16 along K inside the swizzled 128-byte row = +32 bytes = +2 in the
                // (>>4) start-address field
                if constexpr (PAIR)
                  umma_bf16_pair(d_tmem, adesc + static_cast<uint64_t>(k * 2), bdesc + static_cast<uint64_t>(k * 2), idesc,
                                 (kb | k) != 0 ? 1u : 0u);
                else
                  umma_bf16(d_tmem, adesc + static_cast<uint64_t>(k * 2), bdesc + static_cast<uint64_t>(k * 2), idesc,
                            (kb | k) != 0 ? 1u : 0u);
              }
            } else {
              // fp32 emulation: x = hi + mid + lo (three bf16, 24 mantissa bits, exact), and
              // g.q ~ g_hi(q_hi + q_mid + q_lo) + g_mid(q_hi + q_mid) + g_lo q_hi: six bf16 MMAs into one
              // fp32 accumulator; the dropped terms are below 2^-24 of |g||q|.
              constexpr int kTermA[6] = {0, 0, 1, 0, 1, 2};
              constexpr int kTermB[6] = {0, 1, 0, 2, 1, 0};
#pragma unroll
              for (int term = 0; term < 6; ++term) {
                const uint64_t adesc = make_sw128_desc(a_addr + kTermA[term] * kABytes);
                const uint64_t bdesc = make_sw128_desc(a_addr + a_all + kTermB[term] * b_bytes);
#pragma unroll
                for (int k = 0; k < kBlockK / kUmmaK; ++k) {
                  if constexpr (PAIR)
                    umma_bf16_pair(d_tmem, adesc + static_cast<uint64_t>(k * 2), bdesc + static_cast<uint64_t>(k * 2), idesc,
                                   (kb | k | term) != 0 ? 1u : 0u);
                  else
                    umma_bf16(d_tmem, adesc + static_cast<uint64_t>(k * 2), bdesc + static_cast<uint64_t>(k * 2), idesc,
                              (kb | k | term) != 0 ? 1u : 0u);
                }
              }
            }
            // smem slot reusable (in both CTAs of a pair) once these MMAs retire
            if constexpr (PAIR) umma_commit_pair(&sh->empty[stage]); else umma_commit(&sh->empty[stage]);
            // accumulator complete (pair: each CTA's epilogue is told about its own half)
            if (kb == cfg.k_blocks - 1) {
              if constexpr (PAIR) umma_commit_pair(&sh->tmem_full[as]); else umma_commit(&sh->tmem_full[as]);
            }
          }
          __syncwarp();
          if (++stage == static_cast<uint32_t>(cfg.stages)) { stage = 0; phase ^= 1; }
        }
        ++it;
      }
    }
  } else if (warp < EPI_WARPS) {
    // ===== epilogue: TMEM -> registers -> keys / scores =====
    // warp w may read TMEM lanes 32*(w%4) .. +31.  Warps 4-7 take the first half of the 16-column
    // chunks, warps 8-11 the second half of the same rows: two epilogue warps per scheduler hide
    // each other's TMEM-load and shared-memory latencies (with one the 256-query kernel was
    // epilogue-bound: tensor pipe 45 % active, profiles/r01_k2_b256_source.txt).
    const int ew = warp;
    const int quarter = ew & 3, part = ew >> 2;            // EPI_WARPS / 4 warps share a lane quarter
    constexpr int kParts = EPI_WARPS / 4;
    const int r_in_tile = quarter * 32 + lane;
    const int n_chunks = cfg.n_umma / 16;
    const int per_part = (n_chunks + kParts - 1) / kParts;
    const int c_begin = min(part * per_part, n_chunks) * 16;
    const int c_end = min((part + 1) * per_part, n_chunks) * 16;
    const int64_t last_row = p.n_rows - 1;
    const uint32_t tmem_empty_leader = PAIR ? mapa_u32(smem_u32(&sh->tmem_empty[0]), 0) : 0u;
    uint32_t it = 0;
    bool ok = true;
    for (int u = u_begin; u < n_units && ok; u += u_step) {
      const Unit un = unit_of(u);
      if (un.skip) continue;
      const int j = un.j;
      const int t = j * inc;
      // queries of this unit and where their thresholds sit in shared memory
      const int q0 = p.q0 + un.chunk * kMaxQ;
      const int nq = min(p.nq - un.chunk * kMaxQ, kMaxQ);
      const float* thr_s = sh->thr + (PAIR ? un.chunk * kMaxQ : 0);
      const float* thr_raw_s = sh->thr_raw + (PAIR ? un.chunk * kMaxQ : 0);
      const uint32_t as = it & 1, aphase = (it >> 1) & 1;
      const int64_t row = static_cast<int64_t>(t) * kBlockM + r_in_tile;
      // row filter: the warp's 32 rows are one bitmap word (padded to whole tiles, so always readable);
      // loaded before the accumulator wait so that its latency hides behind the MMAs
      uint32_t filter_word = ~0u;
      if constexpr (MODE != kModeScores) {
        if (p.row_filter != nullptr) filter_word = __ldg(p.row_filter + (row >> 5));
      }
      // label-conditioned: this thread's row label (whole tiles are readable), loaded here for the same
      // reason -- one coalesced 128-byte load per warp
      int32_t row_label = 0;
      if constexpr (labeled) row_label = __ldg(p.row_labels + row);
      float s_r = 0.f;   // int8: the row's scale (a tail row past the end reads the last row's)
      if constexpr (I8)
        s_r = i8_row_scale(static_cast<const int8_t*>(p.gallery) + (row <= last_row ? row : last_row) * p.ld, p.dim);
      const int32_t* lab_u = lab_s + (PAIR ? un.chunk * kMaxQ : 0);
      if (!mbar_wait(&sh->tmem_full[as], aphase, &sh->abort, flags)) break;
      tcgen05_fence_after();
      const bool row_ok = row <= last_row && row_allowed(filter_word, row);
      const uint32_t taddr0 = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) +
                              as * static_cast<uint32_t>(cfg.acc_stride);
      bool released = false;
      auto release_accumulator = [&]() {
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) {
          if constexpr (PAIR) mbar_arrive_cluster(tmem_empty_leader + as * 8u);
          else mbar_arrive(&sh->tmem_empty[as]);
        }
      };
      if (!un.valid || (MODE == kModeFilter && cfg.debug_skip_epilogue == 1)) {
        // nothing to read: a duplicate half tile, or mainloop-only timing
      } else if constexpr (MODE == kModeFilter) {
        // One sweep over the accumulator; a passing (column, score) is parked in this thread's
        // private shared-memory stash and the slots are claimed at the end of the tile, four
        // atomicAdds in flight per lane, so a thread waits for ONE L2 round trip per tile instead
        // of one per passing score (the first version did the latter inside the divergent branch:
        // 53 us per tile at 256 queries; a two-sweep ballot variant spent 45 % of its samples
        // re-walking columns: profiles/r01_k2_b64_source.txt).
        uint2* my_stash = sh->stash[ew] + lane;          // [slot][lane]: conflict-free
        uint32_t n_st = 0;
        auto flush = [&]() {
          for (uint32_t i0 = 0; i0 < n_st; i0 += 4) {
            uint2 e[4];
            uint32_t pos[4];
#pragma unroll
            for (int u4 = 0; u4 < 4; ++u4)
              if (i0 + u4 < n_st) {
                e[u4] = my_stash[(i0 + u4) * 32];
                pos[u4] = atomicAdd(p.cnt + q0 + e[u4].x, 1u);
              }
#pragma unroll
            for (int u4 = 0; u4 < 4; ++u4)
              if (i0 + u4 < n_st && pos[u4] < static_cast<uint32_t>(p.cap))
                p.cand[static_cast<int64_t>(q0 + e[u4].x) * p.cap + pos[u4]] =
                    make_key(__uint_as_float(e[u4].y), static_cast<uint32_t>(row));
          }
          n_st = 0;
        };
        auto process16 = [&](const uint32_t (&acc)[16], int c0, uint32_t eligible) {
          // branch-free pass mask for the 16 columns (every taken branch would expose its full
          // latency), then a short loop over the set bits
          uint32_t bits = 0;
          if constexpr (I8) {
            const float4* thr4 = reinterpret_cast<const float4*>(thr_s + c0);
            const float4* aq4 = reinterpret_cast<const float4*>(thr_raw_s + c0);
#pragma unroll
            for (int c4 = 0; c4 < 4; ++c4) {
              const float4 tq = thr4[c4], aq = aq4[c4];
              const float tv[4] = {tq.x, tq.y, tq.z, tq.w}, av[4] = {aq.x, aq.y, aq.z, aq.w};
#pragma unroll
              for (int u4 = 0; u4 < 4; ++u4) {
                const float sc = i8_score(static_cast<int32_t>(acc[c4 * 4 + u4]), av[u4], s_r);
                bits |= (sc < tv[u4]) ? 0u : (1u << (c4 * 4 + u4));
              }
            }
          } else {
          const float4* thr4 = reinterpret_cast<const float4*>((raw_ok ? thr_raw_s : thr_s) + c0);
          const float mul = raw_ok ? 1.0f : p.scale;
#pragma unroll
          for (int c4 = 0; c4 < 4; ++c4) {
            const float4 tq = thr4[c4];
            const float tv[4] = {tq.x, tq.y, tq.z, tq.w};
#pragma unroll
            for (int u4 = 0; u4 < 4; ++u4) {
              const float a = __uint_as_float(acc[c4 * 4 + u4]);
              bits |= ((raw_ok ? a : a * mul) < tv[u4]) ? 0u : (1u << (c4 * 4 + u4));
            }
          }
          }
          if (!row_ok) bits = 0;
          if constexpr (labeled) bits &= eligible;
          while (bits) {
            const int c = __ffs(bits) - 1;
            bits &= bits - 1;
            uint32_t a = acc[0];
#pragma unroll
            for (int u4 = 1; u4 < 16; ++u4) a = (c == u4) ? acc[u4] : a;
            const float sc = I8 ? i8_score(static_cast<int32_t>(a), thr_raw_s[c0 + c], s_r) : __uint_as_float(a) * p.scale;
            if (sc < thr_s[c0 + c]) continue;        // the exact test
            if (n_st == kStash) flush();
            my_stash[n_st * 32] = make_uint2(static_cast<uint32_t>(c0 + c), __float_as_uint(sc));
            ++n_st;
          }
        };
        // label-conditioned: which of 16 columns this thread's row may be returned for -- four broadcast
        // 16-byte shared loads, like the thresholds; computed BEFORE the accumulator loads, while no
        // accumulator register is live (the 8-warp variants have 80 registers)
        auto label_mask16 = [&](int c0) -> uint32_t {
          uint32_t m = 0;
#pragma unroll
          for (int c4 = 0; c4 < 4; ++c4) {
            const int4 lq = reinterpret_cast<const int4*>(lab_u + c0)[c4];
            const int32_t lv[4] = {lq.x, lq.y, lq.z, lq.w};
#pragma unroll
            for (int u4 = 0; u4 < 4; ++u4) m |= label_ok(row_label, lv[u4], p.label_match) ? (1u << (c4 * 4 + u4)) : 0u;
          }
          return m;
        };
        // the labeled small-pair variant (off by default) reads one 16-column load at a time: with two in
        // flight it spilled; so did the int8 variants of 8 epilogue warps (80 registers), which keep 16 scores live
        constexpr int kColStep = ((labeled && EPI_WARPS == 8 && PAIR) || (I8 && EPI_WARPS == 8)) ? 16 : 32;
        for (int c0 = c_begin; c0 < c_end; c0 += kColStep) {
          uint32_t acc0[16], acc1[16];
          const bool two = kColStep == 32 && c0 + 16 < c_end;     // warp-uniform
          uint32_t elig0 = ~0u, elig1 = ~0u;
          if constexpr (labeled) {
            elig0 = label_mask16(c0);
            if (two) elig1 = label_mask16(c0 + 16);
          }
          __syncwarp();
          tmem_ld16(taddr0 + static_cast<uint32_t>(c0), acc0);
          if (two) tmem_ld16(taddr0 + static_cast<uint32_t>(c0 + 16), acc1);   // both loads in flight
          tmem_ld_wait();
          process16(acc0, c0, elig0);
          if (two) process16(acc1, c0 + 16, elig1);
        }
        // the accumulator is read out: hand it back to the MMA warp BEFORE waiting for the slot
        // atomics of the parked candidates (an L2 round trip that used to sit on the critical path
        // tmem_full -> read-out -> flush -> tmem_empty: the MMA warp waited for tmem_empty on most
        // units, profiles/r01_k2_c5like_pair_summary.txt)
        release_accumulator();
        released = true;
        if (n_st) flush();
      } else {
      for (int c0 = c_begin; c0 < c_end; c0 += 16) {
        uint32_t acc[16];
        __syncwarp();
        tmem_ld16(taddr0 + static_cast<uint32_t>(c0), acc);
        tmem_ld_wait();
        if constexpr (MODE == kModeDense) {
          const int64_t slot = static_cast<int64_t>(j) * kBlockM + r_in_tile;
#pragma unroll
          for (int c = 0; c < 16; ++c) {
            if (c0 + c < nq) {
              const float s = I8 ? i8_score(static_cast<int32_t>(acc[c]), thr_raw_s[c0 + c], s_r)
                                 : __uint_as_float(acc[c]) * p.scale;
              const bool ok = row_ok && (!labeled || label_ok(row_label, lab_u[c0 + c], p.label_match));
              p.cand[static_cast<int64_t>(q0 + c0 + c) * p.cap + slot] =
                  ok ? make_key(s, static_cast<uint32_t>(row)) : 0ull;
            }
          }
        } else {
          if (row_ok) {
#pragma unroll
            for (int c = 0; c < 16; ++c) {
              if (c0 + c < nq)
                p.out_scores[static_cast<int64_t>(q0 + c0 + c) * p.ld_out + row] =
                    I8 ? i8_score(static_cast<int32_t>(acc[c]), thr_raw_s[c0 + c], s_r)
                       : __uint_as_float(acc[c]) * p.scale;
            }
          }
        }
      }
      }
      if (!released) release_accumulator();
      ++it;
    }
  }

  tcgen05_fence_before();
  if constexpr (PAIR) {
    __syncwarp();
    cluster_sync_all();   // neither CTA may retire while its peer can still signal or read it
  } else {
    __syncthreads();
  }
  tcgen05_fence_after();
  if (warp == kAllocWarp) {
    if constexpr (PAIR)
      asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base),
                   "r"(static_cast<uint32_t>(cfg.tmem_cols))
                   : "memory");
    else
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base),
                   "r"(static_cast<uint32_t>(cfg.tmem_cols))
                   : "memory");
  }
}

int scan_mma_split_max_queries() { return getenv("MMRS_K2_NO_PAIR") ? kSplitMaxQ : kSplitPairMaxQ; }
int scan_mma_max_queries() {
  const char* e = getenv("MMRS_K2_QCHUNKS");
  const int c = e ? atoi(e) : kMaxQChunks;
  return kMaxQ * (c >= 1 && c <= kMaxQChunks ? c : kMaxQChunks);
}

// The int8 launches pick among the same variants as the bf16 ones.
template <int EPI, bool PAIR, typename Go>
static cudaError_t go_i8(int mode, bool labeled, Go&& go) {
  switch (mode) {
    case kModeScores: return go(scan_mma_kernel<kModeScores, EPI, PAIR, 1, false, true>);
    case kModeDense:
      return labeled ? go(scan_mma_kernel<kModeDense, EPI, PAIR, 1, true, true>) : go(scan_mma_kernel<kModeDense, EPI, PAIR, 1, false, true>);
    default:
      return labeled ? go(scan_mma_kernel<kModeFilter, EPI, PAIR, 1, true, true>) : go(scan_mma_kernel<kModeFilter, EPI, PAIR, 1, false, true>);
  }
}

// g_plane_rows (split == 3): rows between two gallery planes -- the FULL gallery's row count, also when
// p.gallery / p.n_rows are a row window of plane 0 (range search)
// i8: int8 gallery rows and prepared int8 query rows (q_bf16 holds them, p.ldq bytes apart); p.dim and p.ld
// count bytes.  The tensor maps see each 128-byte k-block as 64 bf16 columns: TMA only moves bytes.
cudaError_t launch_scan_mma(const ScanParams& p, const __nv_bfloat16* q_bf16, int32_t n_q_padded,
                            int mode, int32_t* flags, int sm_count, cudaStream_t stream, int split,
                            int64_t g_plane_rows, bool i8) {
  const int n_qchunks = (p.nq + kMaxQ - 1) / kMaxQ;
  if (p.nq < 1 || n_qchunks > kMaxQChunks) return cudaErrorInvalidValue;
  if (split != 1 && split != 3) return cudaErrorInvalidValue;
  if (i8 && (split != 1 || p.dim % 16 != 0 || p.ld % 16 != 0 || p.ldq % 16 != 0)) return cudaErrorInvalidValue;
  if (split == 3 && p.nq > scan_mma_split_max_queries()) return cudaErrorInvalidValue;
  if (p.n_rows > 0x7fffffffll - kBlockM) return cudaErrorInvalidValue;   // TMA coordinates are int32
  if (p.sched.tile_exc != 0 && p.sched.tile_exc % p.sched.tile_inc != 0) return cudaErrorInvalidValue;
  MmaCfg cfg;
  cfg.n_umma = n_qchunks > 1 ? kMaxQ : (p.nq + 15) / 16 * 16;   // multi-chunk launches: full-width tiles (padded columns never pass)
  const int32_t map_cols = i8 ? p.dim / 2 : p.dim;   // in bf16 columns of 2 bytes
  cfg.k_blocks = (map_cols + kBlockK - 1) / kBlockK;
  cfg.split = split;
  cfg.g_plane_rows = g_plane_rows;
  cfg.q_plane_rows = n_q_padded;
  cfg.n_qchunks = n_qchunks;
  cfg.sticky = 0;
  // Idea: the ring holds about one tile per CTA (8 x 16 KB); its slots turn around once per DRAM latency PLUS
  // the time the MMAs of the slot take, so with more queries the bytes in flight per SM might stop covering the
  // loaded HBM latency (kernel 0.151 ms at 16 queries -> 0.174 at 128, proportional to the SM count).  L2
  // prefetches need no shared-memory slot: request the next unit's tile one unit (~3 us) ahead.
  // MEASURED AND REJECTED (profiles/r02_prefetch_ab.log): with the prefetch on, the 16-query scan slows from
  // 0.151 to 0.211 ms and every other shape by 8-30 %: the extra requests compete with the ring's own loads
  // instead of shortening them.  Off by default; the knob stays for A/B runs.
  cfg.prefetch = getenv("MMRS_K2_PREFETCH") ? atoi(getenv("MMRS_K2_PREFETCH")) : 0;
  cfg.debug_skip_epilogue = getenv("MMRS_K2_DEBUG_SKIP_EPI") ? atoi(getenv("MMRS_K2_DEBUG_SKIP_EPI")) : 0;   // 1: no epilogue, 2: nothing passes
  // Up to 64 queries the CTA is sized so that TWO fit on an SM (<= 113 KB of shared memory, 80
  // registers x 384 threads, <= 256 TMEM columns each): the scans of two searches in flight on
  // different streams then share the HBM stream instead of queueing behind each other, and the
  // short seed/mid scans of one search hide under the long last-phase scan of the other.
  // (65..128 queries used to run this way too, with only two 32 KB ring stages per CTA; as CTA
  // pairs they get eight 24 KB stages: 0.216 vs 0.238 ms per step at 128 queries.)
  int small_max = 64;   // 33..64 queries: 3-4 ring stages per CTA, two CTAs per SM
  if (const char* e = getenv("MMRS_K2_SMALL_MAX")) small_max = atoi(e);
  const bool small = split == 1 && cfg.n_umma <= small_max && getenv("MMRS_K2_BIG_SMEM") == nullptr;
  // MEASURED AND REJECTED (profiles/r02_small_pair_ab.log): 65..128 queries as CTA pairs sized like the small
  // variant ("small pair": 8 epilogue warps, <= 113 KB, 80 registers), so that a pair-mode scan does not own its
  // SMs and the second search in flight runs beside it.  With four 24 KB stages the scan itself slows from 0.158 to
  // 0.183 ms and the step from 0.215 to 0.293 ms at 128 queries (0.210 -> 0.255 at 96; no change at 64).  Off by
  // default (MMRS_K2_SMALL_PAIR_MAX=128 turns it on for A/B runs).
  int small_pair_max = 0;
  if (const char* e = getenv("MMRS_K2_SMALL_PAIR_MAX")) small_pair_max = atoi(e);
  const bool small_pair = !small && split == 1 && n_qchunks == 1 && cfg.n_umma <= small_pair_max &&
                          getenv("MMRS_K2_BIG_SMEM") == nullptr && getenv("MMRS_K2_NO_PAIR") == nullptr;
  // Above that the kernel runs as CTA pairs (cta_group::2, see the file header)
  int pair_min = 64;
  if (const char* e = getenv("MMRS_K2_PAIR_MIN")) pair_min = atoi(e);
  // fp32 emulation: up to 48 queries a single CTA per SM holds three stages of all six planes; beyond that the
  // pair halves the query planes per CTA, so that 100 queries (BASELINE C1) are ONE pass over the gallery
  // planes instead of three (1.49 ms -> one 3 GB stream at 1M x 512, profiles/r02_fp32_bench_*.log)
  const bool pair = small_pair ||
                    (!small && (split == 1 ? cfg.n_umma > pair_min : p.nq > kSplitMaxQ) && getenv("MMRS_K2_NO_PAIR") == nullptr);
  if (pair) cfg.n_umma = (cfg.n_umma + 31) / 32 * 32;   // each CTA stages half the query rows
  int cols = 32;
  while (cols < 2 * cfg.n_umma) cols <<= 1;
  cfg.tmem_cols = cols;
  cfg.acc_stride = cols / 2;
  const int b_rows = pair ? cfg.n_umma / 2 : cfg.n_umma;
  const size_t stage_bytes = split * (static_cast<size_t>(kABytes) + static_cast<size_t>(b_rows) * kBlockK * 2);
  const bool half_sm = small || small_pair;   // footprint of half an SM: two CTAs (of two searches) per SM
  const size_t shared_struct = half_sm ? sizeof(MmaSharedT<1, 8>) : (pair ? sizeof(MmaSharedT<kMaxQChunks>) : sizeof(MmaSharedT<1>));
  // label-conditioned launches add the label tail (the kernel's lab_s); unlabeled ones are sized as before
  const bool labeled = mode != kModeScores && p.row_labels != nullptr;
  const size_t label_tail =
      labeled ? (static_cast<size_t>(label_tail_slots(pair, n_qchunks, cfg.n_umma)) * sizeof(int32_t) + 15) / 16 * 16 : 0;
  const size_t budget =
      (half_sm ? 113 * 1024 : 227 * 1024) - shared_struct - label_tail - 1024 - (half_sm ? 1024 : 0);
  int stages = static_cast<int>(budget / stage_bytes);
  if (stages > kMaxStages) stages = kMaxStages;
  if (stages < 2) return cudaErrorInvalidValue;
  cfg.stages = stages;
  const size_t smem = 1024 + stage_bytes * stages + shared_struct + label_tail;

  CUtensorMap map_g, map_q;
  const int64_t g_map_rows = static_cast<int64_t>(split - 1) * g_plane_rows + p.n_rows;   // = split * n_rows unwindowed
  if (g_map_rows > 0x7fffffffll - kBlockM) return cudaErrorInvalidValue;
  // int8: the inner extent is the codes only, so the scale bytes are never loaded as codes and K2 gets zero
  // fill past dim
  if (!make_map(&map_g, p.gallery, static_cast<uint64_t>(g_map_rows), static_cast<uint64_t>(map_cols),
                static_cast<uint64_t>(i8 ? p.ld / 2 : p.ld), kBlockM))
    return cudaErrorNotSupported;
  if (!make_map(&map_q, q_bf16, static_cast<uint64_t>(split) * n_q_padded, static_cast<uint64_t>(i8 ? map_cols : p.ldq),
                static_cast<uint64_t>(i8 ? p.ldq / 2 : p.ldq), static_cast<uint32_t>(b_rows)))
    return cudaErrorNotSupported;

  const int R = plan_exclusion_ratio(p.sched.tile_inc, p.sched.tile_exc);
  const int n_valid = plan_n_visited(p.sched.n_sel, R);
  if (n_valid < 1) return cudaSuccess;   // nothing to visit
  dim3 grid;
  if (pair) {
    // one pair per TPC; units = (tile pair, query chunk)
    const int n_units = plan_pair_units(n_valid, n_qchunks);
    int pairs = sm_count / 2;
    // Measured and rejected (profiles/r02_hbm_pairs_ab.log): running HBM-bound pair launches on 64 or 56 of the 74
    // TPCs, to leave SMs to the second search in flight, slows the scan in proportion (0.174 -> 0.196 -> 0.218 ms
    // at 128 queries): the scan is bound by bytes in flight per SM, not by HBM alone.  The knob stays for A/B runs.
    int hbm_pairs = 0;
    if (const char* e = getenv("MMRS_K2_HBM_PAIRS")) hbm_pairs = atoi(e);
    if (split == 1 && n_qchunks == 1 && cfg.n_umma <= 128 && n_units >= 8 * pairs && hbm_pairs >= 8 && hbm_pairs < pairs)
      pairs = hbm_pairs;
    if (pairs > n_units) pairs = n_units;
    grid = dim3(2 * pairs, 1);
    // every pair gets at least four tile pairs of its own: the chunks of a tile pair can stay on one pair
    const char* st = getenv("MMRS_K2_STICKY");
    cfg.sticky = (st ? atoi(st) != 0 : true) && n_qchunks > 1 && (n_valid + 1) / 2 >= 4 * pairs;
  } else {
    // 33..64 queries: the small-footprint CTA has only 4 ring stages, so one launch fills both CTA
    // slots of every SM itself (measured: 0.202 vs 0.224 ms per step at 64 queries)
    int ctas_per_sm = (small && cfg.n_umma > 32) ? 2 : 1;
    if (const char* e = getenv("MMRS_K2_CTAS_PER_SM")) ctas_per_sm = atoi(e) == 2 && small ? 2 : 1;
    int gx = sm_count * ctas_per_sm / n_qchunks;
    if (gx > p.sched.n_sel) gx = p.sched.n_sel;
    if (gx < 1) gx = 1;
    grid = dim3(gx, n_qchunks);
  }
  auto go = [&](auto kernel) -> cudaError_t {
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e != cudaSuccess) return e;
    return launch_pdl_cluster(kernel, grid, dim3((kCtrlWarps + (half_sm ? 8 : 16)) * 32), smem, stream, pair ? 2u : 1u,
                              map_g, map_q, p, cfg, flags);
  };
  if (i8) {
    if (small) return go_i8<8, false>(mode, labeled, go);
    if (small_pair) return go_i8<8, true>(mode, labeled, go);
    if (pair) return go_i8<16, true>(mode, labeled, go);
    return go_i8<16, false>(mode, labeled, go);
  }
  if (small) {
    switch (mode) {
      case kModeScores: return go(scan_mma_kernel<kModeScores, 8, false, 1>);
      case kModeDense: return labeled ? go(scan_mma_kernel<kModeDense, 8, false, 1, true>) : go(scan_mma_kernel<kModeDense, 8, false, 1>);
      default: return labeled ? go(scan_mma_kernel<kModeFilter, 8, false, 1, true>) : go(scan_mma_kernel<kModeFilter, 8, false, 1>);
    }
  }
  if (small_pair) {
    switch (mode) {   // 65..128 queries: CTA pairs with the footprint of half an SM
      case kModeScores: return go(scan_mma_kernel<kModeScores, 8, true, 1>);
      case kModeDense: return labeled ? go(scan_mma_kernel<kModeDense, 8, true, 1, true>) : go(scan_mma_kernel<kModeDense, 8, true, 1>);
      default: return labeled ? go(scan_mma_kernel<kModeFilter, 8, true, 1, true>) : go(scan_mma_kernel<kModeFilter, 8, true, 1>);
    }
  }
  if (pair && split == 1) {
    switch (mode) {   // > 128 queries: one CTA per SM, CTA pairs, 16 epilogue warps each
      case kModeScores: return go(scan_mma_kernel<kModeScores, 16, true, 1>);
      case kModeDense: return labeled ? go(scan_mma_kernel<kModeDense, 16, true, 1, true>) : go(scan_mma_kernel<kModeDense, 16, true, 1>);
      default: return labeled ? go(scan_mma_kernel<kModeFilter, 16, true, 1, true>) : go(scan_mma_kernel<kModeFilter, 16, true, 1>);
    }
  }
  if (pair) {
    switch (mode) {   // fp32 emulation, 49..128 queries: CTA pairs, three planes per operand
      case kModeScores: return go(scan_mma_kernel<kModeScores, 16, true, 3>);
      case kModeDense: return labeled ? go(scan_mma_kernel<kModeDense, 16, true, 3, true>) : go(scan_mma_kernel<kModeDense, 16, true, 3>);
      default: return labeled ? go(scan_mma_kernel<kModeFilter, 16, true, 3, true>) : go(scan_mma_kernel<kModeFilter, 16, true, 3>);
    }
  }
  if (split == 3) {
    switch (mode) {   // fp32 emulation, up to 48 queries
      case kModeScores: return go(scan_mma_kernel<kModeScores, 16, false, 3>);
      case kModeDense: return labeled ? go(scan_mma_kernel<kModeDense, 16, false, 3, true>) : go(scan_mma_kernel<kModeDense, 16, false, 3>);
      default: return labeled ? go(scan_mma_kernel<kModeFilter, 16, false, 3, true>) : go(scan_mma_kernel<kModeFilter, 16, false, 3>);
    }
  }
  switch (mode) {   // MMRS_K2_NO_PAIR / MMRS_K2_BIG_SMEM
    case kModeScores: return go(scan_mma_kernel<kModeScores, 16, false, 1>);
    case kModeDense: return labeled ? go(scan_mma_kernel<kModeDense, 16, false, 1, true>) : go(scan_mma_kernel<kModeDense, 16, false, 1>);
    default: return labeled ? go(scan_mma_kernel<kModeFilter, 16, false, 1, true>) : go(scan_mma_kernel<kModeFilter, 16, false, 1>);
  }
}

}  // namespace mmrs
