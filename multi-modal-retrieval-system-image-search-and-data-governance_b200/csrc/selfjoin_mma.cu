// selfjoin_mma.cu -- K5 on tensor cores: bf16 tcgen05 prefilter + exact fp32 recheck.
//
// N(N-1)/2 dot products is a GEMM (5.0e13 pairs at N = 10 M, SURVEY.md section 8d C3), so the
// candidate pass runs on the 5th-gen tensor cores over a bf16 copy of the unit-norm embeddings:
//   S[256 rows i, 256 rows j] = X16[i-blocks] * X16[j-block]^T     (tcgen05.mma.cta_group::2, M=256, N=256)
// by a PAIR of CTAs (one TPC): each CTA stages its own 128-row i-block and half of the j-block,
// CTA 0's MMA warp issues for both, each CTA's 128 x 256 accumulator lands in its own TMEM (less
// operand traffic per SM, see scan_mma.cu); long joins use single CTAs (M=128) instead, see
// sjm_pair_mode.  The epilogue keeps pairs (i < j) with S >= tau - margin.  bf16 keeps 8 significant
// bits, so round-to-nearest moves each element by at most u = 2^-8 of its value, and rounding both rows
// moves their dot product by at most ||a|| ||b - b^|| + ||a - a^|| ||b^|| <= (2u + u^2) ||a|| ||b||
// (Cauchy-Schwarz).  Rows whose elements all sit just above a power of two, 2^e (1 + 0.99 * 2^-8), reach
// 99 % of that bound: 0.0077 for unit rows.  Each fp32 dot product adds at most
// dim * 2^-24 / (1 - dim * 2^-24) ||a|| ||b|| when rounded to nearest: the exact mode's sum that decides
// the pair, and S, whose accumulation order and rounding on the tensor cores are not documented; the
// margin allows dim * 2^-22 for the two.  So with margin >= (2^-7 + 2^-16 + dim * 2^-22) max(1, max ||a||^2)
// (dedup.tc_margin) every pair the exact mode emits survives; the few survivors are then re-scored in
// fp32 with exactly the arithmetic of the exact kernel (selfjoin.cu: one fmaf chain, k ascending),
// which makes the emitted pair set identical to the exact mode's.
//
// Schedule: the upper triangle is cut into panels of 8 j-blocks (2048 rows: 2 MB of bf16 at
// D = 512, L2 resident); inside a panel tiles are numbered j-fastest, so CTAs that run together
// share their A rows and the B panel through L2.  Panels are dealt round-robin to the ranks of a
// multi-GPU run (work per panel grows linearly with its index, so cyclic dealing balances).
#include <stdlib.h>

#include "host.h"
#include "tcgen05_utils.cuh"

namespace mmrs {

constexpr int kSjmThreads = 256;
constexpr int kSjmBM = 128;
constexpr int kSjmBN = 256;
constexpr int kSjmBK = 64;
constexpr int kSjmMaxStages = 6;
constexpr int kSjmPanel = 8;   // j-blocks per panel
constexpr int kSjmABytes = kSjmBM * kSjmBK * 2;
// B rows a CTA stages per k-block: the whole j-block, or half of it in pair mode; ring depth to match
template <bool PAIR> struct SjmCfg {
  static constexpr int kBBytes = (PAIR ? kSjmBN / 2 : kSjmBN) * kSjmBK * 2;
  static constexpr int kStageBytes = kSjmABytes + kBBytes;
  static constexpr int kStages = PAIR ? 6 : 4;
};

struct SjmShared {
  uint64_t full[kSjmMaxStages];
  uint64_t empty[kSjmMaxStages];
  uint64_t tmem_full[2];
  uint64_t tmem_empty[2];
  uint32_t tmem_base;
  volatile uint32_t abort;
};

struct SjmParams {
  int64_t n_rows;
  int32_t k_blocks;
  float thr_lo;                    // tau - margin
  int64_t nbi, nbj;                // number of 128-row i-blocks / 256-row j-blocks
  int32_t n_my_panels;             // panels dealt to this rank: panel_begin + m * panel_stride
  int32_t panel_begin, panel_stride;
  const int64_t* panel_start;      // [n_my_panels + 1] first tile number of each of my panels
  int64_t total_tiles;
  int32_t ib_per_tile;             // i-blocks per work unit: 2 in pair mode, else 1
  int64_t* cand;                   // [cand_cap, 2]
  int64_t cand_cap;
  unsigned long long* cand_count;
  // I8 only: the int8 rows (codes, then the row's scale at byte dim_i8), ld_i8 bytes apart
  const int8_t* rows_i8;
  int64_t ld_i8;
  int32_t dim_i8;
};

// work-unit number -> (first i-block of the unit, j-block); returns false when that i-block lies
// entirely on/below the diagonal.  In pair mode a unit is two i-blocks: if the first is below the
// diagonal so is the second; when only the second is, its CTA computes a tile whose columns all
// fail the epilogue's j > i test.
__device__ __forceinline__ bool sjm_decode(const SjmParams& p, int64_t t, int64_t& ib, int64_t& jb) {
  int lo = 0, hi = p.n_my_panels;           // last m with panel_start[m] <= t
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (p.panel_start[mid] <= t) lo = mid; else hi = mid;
  }
  const int64_t panel = p.panel_begin + static_cast<int64_t>(lo) * p.panel_stride;
  const int64_t u = t - p.panel_start[lo];
  int64_t nj = p.nbj - panel * kSjmPanel;
  if (nj > kSjmPanel) nj = kSjmPanel;
  ib = p.ib_per_tile * (u / nj);
  jb = panel * kSjmPanel + u % nj;
  return jb * kSjmBN + (kSjmBN - 1) > ib * kSjmBM;
}

// The smallest dot >= 1 with i8_score(dot, s_i, s_max) >= tau, or INT32_MAX when none up to |dot|'s bound; for
// tau <= 0 (or NaN) INT32_MIN.  i8_score is non-decreasing in dot and, for dot > 0, in s_j, and a pair with
// dot <= 0 scores <= 0; so with s_max the largest s_j of a j-block, every pair of the block that scores >= tau > 0
// has dot >= this value, and the integer test `dot >= d_min` can only pass pairs the exact test then decides.
__device__ __forceinline__ int32_t i8_min_dot(float s_i, float s_max, float tau, int32_t dim) {
  if (!(tau > 0.f)) return INT32_MIN;
  int32_t lo = 1, hi = 127 * 127 * dim;
  if (!(i8_score(hi, s_i, s_max) >= tau)) return INT32_MAX;
  while (lo < hi) {
    const int32_t mid = lo + (hi - lo) / 2;
    if (i8_score(mid, s_i, s_max) >= tau) hi = mid; else lo = mid + 1;
  }
  return lo;
}

// I8: int8 rows (include/mmrs_b200.h, "int8 galleries"), tcgen05.mma.kind::i8 with s32 accumulators.  The TMA
// maps see each 128-byte k-block as 64 bf16 columns (TMA only moves bytes), K = 32 per MMA: four per k-block, the
// same 32-byte descriptor step as bf16.  The epilogue decides each pair exactly, fl(fl(float(dot) s_i) s_j) >=
// tau with the lower row as the query (scale 1), and writes kept pairs straight to the output (p.cand): no margin,
// no recheck.  Column scales are not staged: each warp reads the j-block's 256 scales once per tile for their
// maximum only, which turns the test into one integer compare per column (i8_min_dot); the few columns that pass
// it read their own s_j through the cache.  Staging all 256 for the exact test would cost a barrier among the
// epilogue warps per tile for values that almost no column needs at a deduplication threshold.
template <bool PAIR, bool I8 = false>
__global__ void __launch_bounds__(kSjmThreads, 1)
selfjoin_mma_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                    const SjmParams p, int32_t* flags) {
  constexpr int kSjmStages = SjmCfg<PAIR>::kStages;
  constexpr int kSjmStageBytes = SjmCfg<PAIR>::kStageBytes;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* ring = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  SjmShared* sh = reinterpret_cast<SjmShared*>(ring + kSjmStages * kSjmStageBytes);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = PAIR ? cluster_ctarank() : 0u;     // 0: pair leader
  // work units of this CTA (pair): pair, pair + n_pairs, ...
  const int64_t pair = PAIR ? blockIdx.x >> 1 : blockIdx.x, n_pairs = PAIR ? gridDim.x >> 1 : gridDim.x;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kSjmStages; ++s) { mbar_init(&sh->full[s], 1); mbar_init(&sh->empty[s], 1); }
    // pair mode: the leader's tmem_empty collects the four epilogue warps of both CTAs
    for (int a = 0; a < 2; ++a) { mbar_init(&sh->tmem_full[a], 1); mbar_init(&sh->tmem_empty[a], PAIR ? 8 : 4); }
    sh->abort = 0;
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&map_a)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&map_b)) : "memory");
  }
  if (warp == 2) {
    if constexpr (PAIR) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&sh->tmem_base)),
                   "r"(512u)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&sh->tmem_base)),
                   "r"(512u)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  tcgen05_fence_before();
  if constexpr (PAIR) {
    __syncwarp();
    cluster_sync_all();   // the peer's barriers exist before anything is signalled across
  } else {
    __syncthreads();
  }
  tcgen05_fence_after();
  const uint32_t tmem_base = sh->tmem_base;

  if (warp == 0) {
    if (lane == 0) {   // ===== TMA producer (both CTAs; bytes are credited to the leader's barrier) =====
      uint32_t stage = 0, phase = 0;
      bool ok = true;
      for (int64_t t = pair; t < p.total_tiles && ok; t += n_pairs) {
        int64_t ib, jb;
        if (!sjm_decode(p, t, ib, jb)) continue;
        const int32_t a_row = static_cast<int32_t>((ib + rank) * kSjmBM);   // past the last block: zero-filled
        const int32_t b_row = static_cast<int32_t>(jb * kSjmBN + rank * (kSjmBN / 2));
        for (int kb = 0; kb < p.k_blocks; ++kb) {
          if (!mbar_wait(&sh->empty[stage], phase ^ 1, &sh->abort, flags)) { ok = false; break; }
          uint8_t* a_dst = ring + static_cast<size_t>(stage) * kSjmStageBytes;
          if constexpr (PAIR) {
            const uint32_t full_leader = mapa_u32(smem_u32(&sh->full[stage]), 0);
            if (rank == 0) mbar_expect_tx(&sh->full[stage], 2 * kSjmStageBytes);
            tma_load_2d_pair(a_dst, &map_a, full_leader, kb * kSjmBK, a_row, kEvictLast);
            tma_load_2d_pair(a_dst + kSjmABytes, &map_b, full_leader, kb * kSjmBK, b_row, kEvictLast);
          } else {
            mbar_expect_tx(&sh->full[stage], kSjmStageBytes);
            tma_load_2d(a_dst, &map_a, &sh->full[stage], kb * kSjmBK, a_row, kEvictLast);
            tma_load_2d(a_dst + kSjmABytes, &map_b, &sh->full[stage], kb * kSjmBK, b_row, kEvictLast);
          }
          if (++stage == kSjmStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer: the leader's whole warp walks the loop, one elected lane issues (descriptors
    // stay in uniform registers; with the loop inside `if (lane == 0)` the issue sequence, not the
    // tensor pipe, set the pace -- see scan_mma.cu) =====
    if (rank == 0) {
      const uint32_t idesc = I8 ? make_idesc_i8(kSjmBN, PAIR ? 256u : 128u) : make_idesc(kSjmBN, PAIR ? 256u : 128u);
      const uint32_t ring_addr = smem_u32(ring);
      uint32_t stage = 0, phase = 0, it = 0;
      bool ok = true;
      for (int64_t t = pair; t < p.total_tiles && ok; t += n_pairs) {
        int64_t ib, jb;
        if (!sjm_decode(p, t, ib, jb)) continue;
        const uint32_t as = it & 1, aphase = (it >> 1) & 1;
        if (!__all_sync(0xffffffffu, mbar_wait(&sh->tmem_empty[as], aphase ^ 1, &sh->abort, flags))) break;
        tcgen05_fence_after();
        const uint32_t d_tmem = tmem_base + as * kSjmBN;
        for (int kb = 0; kb < p.k_blocks; ++kb) {
          if (!__all_sync(0xffffffffu, mbar_wait(&sh->full[stage], phase, &sh->abort, flags))) { ok = false; break; }
          tcgen05_fence_after();
          const uint32_t a_addr = ring_addr + stage * kSjmStageBytes;
          if (elect_one()) {
            const uint64_t adesc = make_sw128_desc(a_addr);
            const uint64_t bdesc = make_sw128_desc(a_addr + kSjmABytes);
#pragma unroll
            for (int k = 0; k < kSjmBK / 16; ++k) {
              if constexpr (I8) {
                if constexpr (PAIR)
                  umma_i8_pair(d_tmem, adesc + static_cast<uint64_t>(k * 2), bdesc + static_cast<uint64_t>(k * 2), idesc,
                               (kb | k) != 0 ? 1u : 0u);
                else
                  umma_i8(d_tmem, adesc + static_cast<uint64_t>(k * 2), bdesc + static_cast<uint64_t>(k * 2), idesc,
                          (kb | k) != 0 ? 1u : 0u);
              } else if constexpr (PAIR)
                umma_bf16_pair(d_tmem, adesc + static_cast<uint64_t>(k * 2), bdesc + static_cast<uint64_t>(k * 2), idesc,
                               (kb | k) != 0 ? 1u : 0u);
              else
                umma_bf16(d_tmem, adesc + static_cast<uint64_t>(k * 2), bdesc + static_cast<uint64_t>(k * 2), idesc,
                          (kb | k) != 0 ? 1u : 0u);
            }
            if constexpr (PAIR) umma_commit_pair(&sh->empty[stage]); else umma_commit(&sh->empty[stage]);
            if (kb == p.k_blocks - 1) {
              if constexpr (PAIR) umma_commit_pair(&sh->tmem_full[as]); else umma_commit(&sh->tmem_full[as]);
            }
          }
          __syncwarp();
          if (++stage == kSjmStages) { stage = 0; phase ^= 1; }
        }
        ++it;
      }
    }
  } else if (warp >= 4) {
    // ===== epilogue: keep (i < j) with S >= tau - margin (I8: with the exact score >= tau) =====
    const int ew = warp - 4;
    const uint32_t tmem_empty_leader = PAIR ? mapa_u32(smem_u32(&sh->tmem_empty[0]), 0) : 0u;
    uint32_t it = 0;
    for (int64_t t = pair; t < p.total_tiles; t += n_pairs) {
      int64_t ib, jb;
      if (!sjm_decode(p, t, ib, jb)) continue;
      const uint32_t as = it & 1, aphase = (it >> 1) & 1;
      if (!mbar_wait(&sh->tmem_full[as], aphase, &sh->abort, flags)) break;
      tcgen05_fence_after();
      const int64_t i = (ib + rank) * kSjmBM + ew * 32 + lane;
      const int64_t j0 = jb * kSjmBN;
      const uint32_t taddr0 = tmem_base + (static_cast<uint32_t>(ew * 32) << 16) + as * kSjmBN;
      // a warp whose 32 rows all lie at or beyond the j-block's last column has nothing to keep
      if ((ib + rank) * kSjmBM + ew * 32 < j0 + kSjmBN - 1) {
        float s_i = 0.f;
        int32_t d_min = 0;
        if constexpr (I8) {
          float s_max = 0.f;
#pragma unroll
          for (int m = 0; m < kSjmBN / 32; ++m) {
            const int64_t j = j0 + m * 32 + lane;
            if (j < p.n_rows) s_max = fmaxf(s_max, i8_row_scale(p.rows_i8 + j * p.ld_i8, p.dim_i8));
          }
#pragma unroll
          for (int o = 16; o >= 1; o >>= 1) s_max = fmaxf(s_max, __shfl_xor_sync(0xffffffffu, s_max, o));
          if (i < p.n_rows) s_i = i8_row_scale(p.rows_i8 + i * p.ld_i8, p.dim_i8);
          d_min = i8_min_dot(s_i, s_max, p.thr_lo, p.dim_i8);
        }
        for (int c0 = 0; c0 < kSjmBN; c0 += 16) {
          uint32_t acc[16];
          __syncwarp();
          tmem_ld16(taddr0 + static_cast<uint32_t>(c0), acc);
          tmem_ld_wait();
          uint32_t bits = 0;
#pragma unroll
          for (int c = 0; c < 16; ++c) {
            if constexpr (I8) {
              const int32_t dot = static_cast<int32_t>(acc[c]);
              const int64_t j = j0 + c0 + c;
              if (dot >= d_min && j > i && j < p.n_rows &&
                  i8_score(dot, s_i, i8_row_scale(p.rows_i8 + j * p.ld_i8, p.dim_i8)) >= p.thr_lo)
                bits |= 1u << c;
            } else {
              bits |= (__uint_as_float(acc[c]) >= p.thr_lo) ? (1u << c) : 0u;
            }
          }
          while (bits) {
            const int c = __ffs(bits) - 1;
            bits &= bits - 1;
            const int64_t j = j0 + c0 + c;
            if (j > i && j < p.n_rows) {   // i < j < n_rows
              const unsigned long long pos = atomicAdd(p.cand_count, 1ull);
              if (pos < static_cast<unsigned long long>(p.cand_cap)) {
                p.cand[2 * pos] = i;
                p.cand[2 * pos + 1] = j;
              }
            }
          }
        }
      }
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) {
        if constexpr (PAIR) mbar_arrive_cluster(tmem_empty_leader + as * 8u);
        else mbar_arrive(&sh->tmem_empty[as]);
      }
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
  if (warp == 2) {
    if constexpr (PAIR)
      asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    else
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
  }
}

// Exact fp32 re-score of the candidates: the same single fmaf chain, k ascending, as
// selfjoin_f32_kernel, so both modes take bit-identical decisions.  T = __nv_bfloat16: the rows of a bf16
// gallery, each element widened to fp32 (exactly) before the same chain -- the exact join of those rows in fp32.
template <typename T>
__global__ void __launch_bounds__(256) selfjoin_recheck_kernel(const int64_t* __restrict__ cand, int64_t n_cand,
                                                               const T* __restrict__ emb, int64_t ld, int32_t dim,
                                                               float threshold, int64_t* __restrict__ out_pairs,
                                                               int64_t capacity, unsigned long long* out_count) {
  const int64_t c = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (c >= n_cand) return;
  const int64_t i = cand[2 * c], j = cand[2 * c + 1];
  float acc = 0.f;
  if constexpr (sizeof(T) == 4) {
    const float4* a = reinterpret_cast<const float4*>(emb + i * ld);
    const float4* b = reinterpret_cast<const float4*>(emb + j * ld);
    for (int k = 0; k < dim / 4; ++k) {
      const float4 x = a[k], y = b[k];
      acc = fmaf(x.x, y.x, acc); acc = fmaf(x.y, y.y, acc);
      acc = fmaf(x.z, y.z, acc); acc = fmaf(x.w, y.w, acc);
    }
  } else {
    const uint4* a = reinterpret_cast<const uint4*>(emb + i * ld);
    const uint4* b = reinterpret_cast<const uint4*>(emb + j * ld);
    for (int k = 0; k < dim / 8; ++k) {   // 8 bf16 per 16-byte load
      const uint4 x = a[k], y = b[k];
      const __nv_bfloat162* x2 = reinterpret_cast<const __nv_bfloat162*>(&x);
      const __nv_bfloat162* y2 = reinterpret_cast<const __nv_bfloat162*>(&y);
#pragma unroll
      for (int h = 0; h < 4; ++h) {
        const float2 u = __bfloat1622float2(x2[h]), v = __bfloat1622float2(y2[h]);
        acc = fmaf(u.x, v.x, acc); acc = fmaf(u.y, v.y, acc);
      }
    }
  }
  if (acc >= threshold) {
    const unsigned long long pos = atomicAdd(out_count, 1ull);
    if (pos < static_cast<unsigned long long>(capacity)) {
      out_pairs[2 * pos] = i;
      out_pairs[2 * pos + 1] = j;
    }
  }
}

// ---- host side -------------------------------------------------------------------------------------
// Fills h_panel_start (n_my_panels + 1 entries) and returns the launch parameters.
// CTA pairs or single CTAs?  Pairs keep the tensor pipe busier (+11-14 % on joins that finish within
// ~0.1 s), but a long join runs against the board's power cap, where what counts is energy per
// flop and the single-CTA kernel came out 5 % ahead (same-box A/B on one rank's share of C3:
// 5.91 s vs 6.20-6.31 s, profiles/r01_selfjoin_ab.log).  So: pairs below ~0.12 s of estimated work.
static bool sjm_pair_mode(int64_t n_rows, int32_t dim, int32_t world) {
  if (const char* e = getenv("MMRS_SJ_PAIR")) return atoi(e) != 0;
  const double flops = static_cast<double>(dim) * static_cast<double>(n_rows) * static_cast<double>(n_rows) /
                       static_cast<double>(world > 0 ? world : 1);
  return flops < 1.44e14;
}

static int64_t sjm_plan(int64_t n_rows, int32_t rank, int32_t world, bool pair, int64_t* h_panel_start, int32_t max_panels,
                        int32_t* n_my_panels) {
  const int64_t nbi = (n_rows + kSjmBM - 1) / kSjmBM, nbj = (n_rows + kSjmBN - 1) / kSjmBN;
  const int64_t n_panels = (nbj + kSjmPanel - 1) / kSjmPanel;
  int32_t m = 0;
  int64_t tiles = 0;
  for (int64_t pnl = rank; pnl < n_panels && m < max_panels; pnl += world, ++m) {
    if (h_panel_start) h_panel_start[m] = tiles;
    int64_t ni = 2 * kSjmPanel * (pnl + 1);
    if (ni > nbi) ni = nbi;
    int64_t nj = nbj - pnl * kSjmPanel;
    if (nj > kSjmPanel) nj = kSjmPanel;
    tiles += (pair ? (ni + 1) / 2 : ni) * nj;   // a CTA pair takes two i-blocks at a time
  }
  if (h_panel_start) h_panel_start[m] = tiles;
  *n_my_panels = m;
  return tiles;
}

static int64_t sjm_max_panels(int64_t n_rows) {
  const int64_t nbj = (n_rows + kSjmBN - 1) / kSjmBN;
  return (nbj + kSjmPanel - 1) / kSjmPanel;
}

// rows: bf16 [n_rows, ld] (ld in elements), or with i8 int8 rows of ld bytes (codes [dim], then the scale)
static cudaError_t launch_selfjoin_mma(const void* rows, bool i8, int64_t n_rows, int32_t dim, int64_t ld,
                                       float thr_lo, int32_t rank, int32_t world, bool pair, const int64_t* d_panel_start,
                                       int32_t n_my_panels, int64_t total_tiles, int64_t* cand, int64_t cand_cap,
                                       unsigned long long* cand_count, int32_t* flags, int sm_count,
                                       cudaStream_t stream) {
  if (total_tiles <= 0) return cudaSuccess;
  if (n_rows > 0x7fffffffll - kSjmBN) return cudaErrorInvalidValue;
  SjmParams p{};
  p.n_rows = n_rows;
  const int32_t map_cols = i8 ? dim / 2 : dim;   // in bf16 columns of 2 bytes: TMA only moves bytes
  p.k_blocks = (map_cols + kSjmBK - 1) / kSjmBK;
  p.thr_lo = thr_lo;
  p.nbi = (n_rows + kSjmBM - 1) / kSjmBM;
  p.nbj = (n_rows + kSjmBN - 1) / kSjmBN;
  p.n_my_panels = n_my_panels;
  p.panel_begin = rank;
  p.panel_stride = world;
  p.panel_start = d_panel_start;
  p.total_tiles = total_tiles;
  p.ib_per_tile = pair ? 2 : 1;
  p.cand = cand; p.cand_cap = cand_cap; p.cand_count = cand_count;
  if (i8) { p.rows_i8 = static_cast<const int8_t*>(rows); p.ld_i8 = ld; p.dim_i8 = dim; }
  // int8: the inner extent is the codes only, so the scale bytes are never loaded as codes
  const uint64_t map_ld = static_cast<uint64_t>(i8 ? ld / 2 : ld);
  CUtensorMap map_a, map_b;
  if (!make_map(&map_a, rows, static_cast<uint64_t>(n_rows), static_cast<uint64_t>(map_cols), map_ld, kSjmBM))
    return cudaErrorNotSupported;
  if (!make_map(&map_b, rows, static_cast<uint64_t>(n_rows), static_cast<uint64_t>(map_cols), map_ld, pair ? kSjmBN / 2 : kSjmBN))
    return cudaErrorNotSupported;
  const size_t smem = 1024 + sizeof(SjmShared) +
                      (pair ? static_cast<size_t>(SjmCfg<true>::kStages) * SjmCfg<true>::kStageBytes
                            : static_cast<size_t>(SjmCfg<false>::kStages) * SjmCfg<false>::kStageBytes);
  auto kernel = i8 ? (pair ? selfjoin_mma_kernel<true, true> : selfjoin_mma_kernel<false, true>)
                  : (pair ? selfjoin_mma_kernel<true> : selfjoin_mma_kernel<false>);
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
  if (e != cudaSuccess) return e;
  int64_t units = pair ? sm_count / 2 : sm_count;          // one CTA (pair) per SM (TPC)
  if (units > total_tiles) units = total_tiles;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(static_cast<unsigned>(pair ? 2 * units : units)); cfg.blockDim = dim3(kSjmThreads);
  cfg.dynamicSmemBytes = smem; cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = pair ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, map_a, map_b, p, flags);
}

template <typename T>
static cudaError_t launch_selfjoin_recheck(const int64_t* cand, int64_t n_cand, const T* emb, int64_t ld, int32_t dim,
                                           float threshold, int64_t* out_pairs, int64_t capacity,
                                           unsigned long long* out_count, cudaStream_t stream) {
  if (n_cand <= 0) return cudaSuccess;
  selfjoin_recheck_kernel<T><<<static_cast<int>((n_cand + 255) / 256), 256, 0, stream>>>(
      cand, n_cand, emb, ld, dim, threshold, out_pairs, capacity, out_count);
  return cudaGetLastError();
}


// The workspace of mmrs_selfjoin_pairs_tc / _stored: the flag word, the two counts, the panel starts, the candidate
// pairs (none for an int8 join, whose kernel writes the pairs themselves).
struct SjmWorkspace {
  int32_t* flags;
  unsigned long long* counts;   // [0] pairs, [1] candidates
  int64_t* panel_start;         // [max_panels + 1]
  int64_t* cand;                // [cand_capacity, 2]
};

static SjmWorkspace carve_sjm(Carver& c, int64_t n_rows, int64_t cand_capacity) {
  SjmWorkspace w;
  w.flags = c.take<int32_t>(sizeof(int32_t));
  w.counts = c.take<unsigned long long>(2 * sizeof(unsigned long long));
  w.panel_start = c.take<int64_t>(static_cast<size_t>(sjm_max_panels(n_rows) + 1) * sizeof(int64_t));
  w.cand = c.take<int64_t>(static_cast<size_t>(cand_capacity) * 2 * sizeof(int64_t));
  return w;
}

// The rest of mmrs_selfjoin_pairs_tc / _stored once the arguments are checked: the tensor-core pass over `rows`
// (bf16, or int8 with exact decisions written straight to the output), then for bf16 the recheck of the candidates
// from `src` (fp32, or with src_bf16 the bf16 rows themselves).
static int selfjoin_tc_run(const void* rows, int64_t ld, bool i8, const void* src, bool src_bf16, int64_t ld_src,
                           int64_t n_rows, int32_t dim, float threshold, float margin, int32_t rank, int32_t world,
                           int64_t* d_out_pairs, int64_t capacity, int64_t* d_out_count, int64_t cand_capacity,
                           void* d_workspace, int sm_count, cudaStream_t stream) {
  Carver c(d_workspace);
  const SjmWorkspace w = carve_sjm(c, n_rows, i8 ? 0 : cand_capacity);
  const int64_t max_panels = sjm_max_panels(n_rows);

  std::vector<int64_t> h_panel(static_cast<size_t>(max_panels) + 1);
  int32_t n_my = 0;
  const bool pair = sjm_pair_mode(n_rows, dim, world);
  const int64_t tiles = sjm_plan(n_rows, rank, world, pair, h_panel.data(), static_cast<int32_t>(max_panels), &n_my);
  MMRS_CUDA(cudaMemsetAsync(w.flags, 0, 512, stream));   // the flag word and the counts: the first two 256-byte pieces
  MMRS_CUDA(cudaMemcpyAsync(w.panel_start, h_panel.data(), static_cast<size_t>(n_my + 1) * sizeof(int64_t),
                            cudaMemcpyHostToDevice, stream));
  MMRS_CUDA(cudaStreamSynchronize(stream));   // h_panel is pageable and goes out of scope
  // int8: the kernel's "candidates" are the pairs, counted in [1] like the bf16 pass's candidates
  MMRS_LAUNCH(launch_selfjoin_mma(rows, i8, n_rows, dim, ld, threshold - margin, rank, world, pair, w.panel_start, n_my,
                                  tiles, i8 ? d_out_pairs : w.cand, i8 ? capacity : cand_capacity, w.counts + 1,
                                  w.flags, sm_count, stream));
  int32_t* h = pinned_status();
  if (!h) return fail(MMRS_ERR_CUDA, "cudaHostAlloc for the status word failed");
  int64_t* h64 = reinterpret_cast<int64_t*>(h);      // 32 bytes: [0] pairs, [1] candidates, [2] flags
  MMRS_CUDA(cudaMemcpyAsync(h64 + 1, w.counts + 1, sizeof(int64_t), cudaMemcpyDeviceToHost, stream));
  MMRS_CUDA(cudaMemcpyAsync(h64 + 2, w.flags, sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
  MMRS_CUDA(cudaStreamSynchronize(stream));
  if (h[4] & kFlagWatchdog) return fail(MMRS_ERR_INTERNAL, "self-join pipeline watchdog fired");
  const int64_t n_cand = h64[1];
  if (i8) {
    h64[0] = n_cand;
    MMRS_CUDA(cudaMemcpyAsync(w.counts, w.counts + 1, sizeof(int64_t), cudaMemcpyDeviceToDevice, stream));
  } else {
    h64[0] = 0;
    if (n_cand <= cand_capacity) {
      if (src_bf16)
        MMRS_LAUNCH(launch_selfjoin_recheck(w.cand, n_cand, static_cast<const __nv_bfloat16*>(src), ld_src, dim, threshold,
                                            d_out_pairs, capacity, w.counts, stream));
      else
        MMRS_LAUNCH(launch_selfjoin_recheck(w.cand, n_cand, static_cast<const float*>(src), ld_src, dim, threshold,
                                            d_out_pairs, capacity, w.counts, stream));
      MMRS_CUDA(cudaMemcpyAsync(h64, w.counts, sizeof(int64_t), cudaMemcpyDeviceToHost, stream));
    }
  }
  MMRS_CUDA(cudaMemcpyAsync(d_out_count, w.counts, 2 * sizeof(int64_t), cudaMemcpyDeviceToDevice, stream));
  MMRS_CUDA(cudaStreamSynchronize(stream));
  if (!i8 && n_cand > cand_capacity)
    return fail(MMRS_ERR_CAPACITY, "%lld candidate pairs, candidate capacity %lld", (long long)n_cand,
                (long long)cand_capacity);
  if (h64[0] > capacity)
    return fail(MMRS_ERR_CAPACITY, "%lld pairs found, capacity %lld", (long long)h64[0], (long long)capacity);
  return MMRS_OK;
}

}  // namespace mmrs

using namespace mmrs;

extern "C" {

size_t mmrs_selfjoin_tc_workspace_bytes(int64_t n_rows, int64_t cand_capacity) {
  if (n_rows < 1) n_rows = 1;
  if (cand_capacity < 1) cand_capacity = 1;
  Carver c(nullptr);
  carve_sjm(c, n_rows, cand_capacity);
  return c.off;
}

int mmrs_selfjoin_pairs_tc(const float* d_emb_f32, int64_t ld_f32, const void* d_emb_bf16, int64_t ld_bf16,
                           int64_t n_rows, int32_t dim, float threshold, float margin, int32_t rank,
                           int32_t world, int64_t* d_out_pairs, int64_t capacity, int64_t* d_out_count,
                           int64_t cand_capacity, void* d_workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceInfo dev;
  int rc = current_device(&dev);
  if (rc != MMRS_OK) return rc;
  rc = check_matrix(d_emb_f32, n_rows, dim, ld_f32, MMRS_DTYPE_F32, "fp32 embeddings");
  if (rc != MMRS_OK) return rc;
  rc = check_matrix(d_emb_bf16, n_rows, dim, ld_bf16, MMRS_DTYPE_BF16, "bf16 embeddings");
  if (rc != MMRS_OK) return rc;
  if (!(margin >= 0.f) || world < 1 || rank < 0 || rank >= world)
    return fail(MMRS_ERR_ARG, "bad margin / rank / world");
  if (capacity < 0 || cand_capacity < 1 || (capacity > 0 && !d_out_pairs) || !d_out_count)
    return fail(MMRS_ERR_ARG, "bad output arguments");
  rc = check_workspace(d_workspace, workspace_bytes, mmrs_selfjoin_tc_workspace_bytes(n_rows, cand_capacity));
  if (rc != MMRS_OK) return rc;
  return selfjoin_tc_run(d_emb_bf16, ld_bf16, false, d_emb_f32, false, ld_f32, n_rows, dim, threshold, margin, rank,
                         world, d_out_pairs, capacity, d_out_count, cand_capacity, d_workspace, dev.sm_count, stream);
}

size_t mmrs_selfjoin_stored_workspace_bytes(int64_t n_rows, int32_t dtype, int64_t cand_capacity) {
  if (n_rows < 1) n_rows = 1;
  if (cand_capacity < 1) cand_capacity = 1;
  Carver c(nullptr);
  carve_sjm(c, n_rows, dtype == MMRS_DTYPE_I8 ? 0 : cand_capacity);
  return c.off;
}

int mmrs_selfjoin_pairs_stored(const void* d_rows, int32_t dtype, int64_t ld, int64_t n_rows, int32_t dim,
                               float threshold, float margin, int32_t rank, int32_t world, int64_t* d_out_pairs,
                               int64_t capacity, int64_t* d_out_count, int64_t cand_capacity, void* d_workspace,
                               size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceInfo dev;
  int rc = current_device(&dev);
  if (rc != MMRS_OK) return rc;
  if (dtype != MMRS_DTYPE_BF16 && dtype != MMRS_DTYPE_I8)
    return fail(MMRS_ERR_ARG, "the stored-format self-join takes bf16 or int8 rows, not dtype %d", dtype);
  const bool i8 = dtype == MMRS_DTYPE_I8;
  rc = check_matrix(d_rows, n_rows, dim, ld, dtype, i8 ? "int8 rows" : "bf16 rows");
  if (rc != MMRS_OK) return rc;
  if (i8 && margin != 0.f) return fail(MMRS_ERR_ARG, "the int8 join decides every pair exactly: margin must be 0");
  if (i8 && dim > 131072) return fail(MMRS_ERR_ARG, "int8 dim %d: the join's int32 dot products allow 131072", dim);
  if (!(margin >= 0.f) || world < 1 || rank < 0 || rank >= world)
    return fail(MMRS_ERR_ARG, "bad margin / rank / world");
  if (capacity < 0 || (!i8 && cand_capacity < 1) || (capacity > 0 && !d_out_pairs) || !d_out_count)
    return fail(MMRS_ERR_ARG, "bad output arguments");
  rc = check_workspace(d_workspace, workspace_bytes, mmrs_selfjoin_stored_workspace_bytes(n_rows, dtype, cand_capacity));
  if (rc != MMRS_OK) return rc;
  return selfjoin_tc_run(d_rows, ld, i8, d_rows, true, ld, n_rows, dim, threshold, margin, rank, world, d_out_pairs,
                         capacity, d_out_count, cand_capacity, d_workspace, dev.sm_count, stream);
}

}  // extern "C"
