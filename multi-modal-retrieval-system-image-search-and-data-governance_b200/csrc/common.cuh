// common.cuh -- shared device/host helpers for the mmrs_b200 kernels (sm_100a only).
#pragma once

#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/mmrs_b200.h"

namespace mmrs {

// Every scan kernel walks the gallery in row tiles of this many rows; the phase
// schedule (plan.h) is expressed in tiles.
constexpr int kTileRows = 128;

// Status bits a kernel can raise in the device-side flag word.
constexpr int kFlagOverflow = 1;      // a candidate list outgrew its capacity
constexpr int kFlagZeroNorm = 2;      // normalize_queries and ||q|| == 0
constexpr int kFlagShort = 4;         // fewer than k candidates reached a select (bug guard)
constexpr int kFlagWatchdog = 8;      // an mbarrier wait timed out (K2 debug guard)
constexpr int kFlagGatherTimeout = 16;  // fused all-gather: a peer rank's flag did not arrive in time
constexpr int kFlagNonFinite = 32;      // int8 mode: a query row holds a NaN or an infinity
constexpr int kFlagBadCandidate = 64;   // refine: a candidate row outside [-1, n_rows)

// Status bits of the duplicate resolve (dedup_resolve.cu), in its own status word.
constexpr int kResolveOrderRange = 1;   // an order id outside [0, n_items)
constexpr int kResolveOrderRepeat = 2;  // an id appears twice in the order
constexpr int kResolvePairRange = 4;    // a pair id outside [0, n_items)

// ---- order-preserving (score, row) -> u64 key ---------------------------------------------
// Larger key == better match: higher score first, then LOWER row index.  Keys are unique
// because row indices are, so "the k largest keys" is a deterministic set and order -- this is
// the tie rule of SURVEY.md H1 (score desc, index asc == stable descending sort).
__host__ __device__ __forceinline__ uint32_t orderable_from_float(float f) {
#ifdef __CUDA_ARCH__
  uint32_t u = __float_as_uint(f);
#else
  union { float f; uint32_t u; } c; c.f = f; uint32_t u = c.u;
#endif
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__host__ __device__ __forceinline__ float float_from_orderable(uint32_t o) {
  uint32_t u = (o & 0x80000000u) ? (o & 0x7fffffffu) : ~o;
#ifdef __CUDA_ARCH__
  return __uint_as_float(u);
#else
  union { float f; uint32_t u; } c; c.u = u; return c.f;
#endif
}
__host__ __device__ __forceinline__ uint64_t make_key(float score, uint32_t row) {
  score += 0.0f;  // -0.0 -> +0.0: the two compare equal, so they must tie (and fall to the index)
  return (static_cast<uint64_t>(orderable_from_float(score)) << 32) | static_cast<uint64_t>(~row);
}
__host__ __device__ __forceinline__ float key_score(uint64_t key) {
  return float_from_orderable(static_cast<uint32_t>(key >> 32));
}
__host__ __device__ __forceinline__ uint32_t key_row(uint64_t key) {
  return ~static_cast<uint32_t>(key);
}

// ---- int8 galleries (include/mmrs_b200.h, "int8 galleries") ----------------------------------------
// The one score formula of every int8 path: fl(fl(float(dot) * a_q) * s_r), -0.0 returned as +0.0.
// dot is the exact int32 code product; a_q = fl(s_q * scale) is taken once per query.
__device__ __forceinline__ float i8_score(int32_t dot, float a_q, float s_r) {
  return __fmul_rn(__fmul_rn(__int2float_rn(dot), a_q), s_r) + 0.0f;
}
// the row's fp32 scale sits at byte `dim` of the row (dim = the padded code count)
__device__ __forceinline__ float i8_row_scale(const void* row, int32_t dim) {
  return __ldg(reinterpret_cast<const float*>(static_cast<const int8_t*>(row) + dim));
}

// ---- streaming loads -------------------------------------------------------------------------
__device__ __forceinline__ uint4 ldg_stream_16B(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}

// ---- programmatic dependent launch ------------------------------------------------------------------
// A search is a chain of short kernels.  Each one lets its successor start launching right away
// (launch_dependents) and blocks on its predecessor's results only after its own prologue
// (griddepcontrol.wait returns once the preceding grid has completed and its writes are visible),
// so launch latency, TMEM allocation and barrier set-up overlap the predecessor's tail.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

bool pdl_enabled();   // api.cu: MMRS_NO_PDL=1 turns the launch attribute off

// cluster_x > 1: the grid is launched as thread-block clusters of that many CTAs along x
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl_cluster(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem,
                                      cudaStream_t stream, unsigned cluster_x, Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  unsigned n = 0;
  if (cluster_x > 1) {
    attr[n].id = cudaLaunchAttributeClusterDimension;
    attr[n].val.clusterDim.x = cluster_x; attr[n].val.clusterDim.y = 1; attr[n].val.clusterDim.z = 1;
    ++n;
  }
  if (pdl_enabled()) {
    attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[n].val.programmaticStreamSerializationAllowed = 1;
    ++n;
  }
  cfg.attrs = attr;
  cfg.numAttrs = n;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem,
                              cudaStream_t stream, Args&&... args) {
  return launch_pdl_cluster(kernel, grid, block, smem, stream, 1u, static_cast<Args&&>(args)...);
}

// ---- flags exchanged between GPUs (system scope) ----------------------------------------------------
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_relaxed_sys(uint32_t* p, uint32_t v) {   // after a fence.sys: fence + relaxed store = release
  asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint64_t global_timer_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}
// Wait until flags[i] >= want for every i in [0, n).  Bounded by wall time: a peer that never
// arrives (a dead rank) must end this kernel with a status flag, not hang the GPU.  A peer that is
// merely late is waited for -- no rank can decide on its own to drop the batch (the others would
// not know), so the bound is generous (MMRS_GATHER_TIMEOUT_MS, default 20 s).
__device__ __forceinline__ void wait_all_ge(const uint32_t* flags, int n, uint32_t want, int32_t* status,
                                            uint64_t timeout_ns) {
  const uint64_t t0 = global_timer_ns();
  for (int i = 0; i < n; ++i) {
    uint32_t spins = 0;
    while (static_cast<int32_t>(ld_acquire_sys(flags + i) - want) < 0) {
      if ((++spins & 1023u) == 0 && global_timer_ns() - t0 > timeout_ns) {
        atomicOr(status, kFlagGatherTimeout);
        return;
      }
      __nanosleep(64);
    }
  }
}

// ---- epilogue modes of the scan kernels ---------------------------------------------------
enum ScanMode : int {
  kModeScores = 0,  // write fp32 scores to out[q, row]                  (full_scores)
  kModeDense = 1,   // write every key at a fixed slot, no atomics         (seed phase)
  kModeFilter = 2   // append keys whose score passes thr[q] (atomic slot) (later phases)
};

// Which tiles a launch covers: t = j * tile_inc for j in [0, n_sel), skipping t with
// t % tile_exc == 0 when tile_exc != 0 (those were covered by an earlier phase).
struct TileSchedule {
  int32_t n_tiles;   // ceil(n_rows / kTileRows)
  int32_t tile_inc;
  int32_t tile_exc;
  int32_t n_sel;     // ceil(n_tiles / tile_inc)
};

struct ScanParams {
  const void* gallery;    // [n_rows, ld] T
  int64_t n_rows;
  int64_t ld;             // elements
  int32_t dim;
  int32_t label_match;    // label-conditioned search: MMRS_LABEL_SAME / MMRS_LABEL_OTHER (see row_labels)
  const float* queries;   // prepared fp32 queries [*, ldq] (normalised, bf16-rounded in bf16 mode); int8 mode:
                          // the prepared int8 query rows in the gallery's row format (s_q at byte dim), ldq bytes
  int32_t ldq;
  int32_t q0;             // first query of this pass
  int32_t nq;             // queries in this pass (<= template QN)
  float scale;
  TileSchedule sched;
  // kModeScores.  The label pointers of a label-conditioned dense / filter launch share their storage:
  // ScanParams keeps the 128-byte layout of the unlabeled search (growing it changed ptxas's register
  // allocation of unlabeled kernels, DESIGN.md section 4).
  //   row_labels: one label per local row, padded to whole tiles (nullptr = unlabeled)
  //   query_labels: indexed by absolute query id
  // A pair (row, query) is eligible iff label_ok (below).  Only the kernels' LABELED instantiations
  // read them; the launchers pick those when row_labels != nullptr in kModeDense / kModeFilter.
  union { float* out_scores; const int32_t* row_labels; };
  union { int64_t ld_out; const int32_t* query_labels; };
  // kModeDense / kModeFilter
  uint64_t* cand;         // [n_queries, cap] keys
  uint32_t* cnt;          // [n_queries]
  const float* thr;       // [n_queries] current lower bound on the k-th best score
  int32_t cap;
  // kModeDense / kModeFilter, optional: allow-list bitmap over the rows (bit r & 31 of word r >> 5),
  // zero-padded to whole tiles; an excluded row is key 0 in dense mode and never appended.
  // nullptr = every row.  kModeScores ignores it.
  const uint32_t* row_filter;
};
static_assert(sizeof(ScanParams) == 128, "the unlabeled kernels were tuned with this parameter layout");

__device__ __forceinline__ bool row_allowed(uint32_t word, int64_t row) { return (word >> (row & 31)) & 1u; }
// query label < 0: every row; otherwise same: row label == query label, other: !=
__device__ __forceinline__ bool label_ok(int32_t row_label, int32_t query_label, int32_t match_other) {
  return query_label < 0 || ((row_label == query_label) != (match_other != 0));
}

struct SelectParams {
  uint64_t* cand;         // [n_queries, cap]
  uint32_t* cnt;          // [n_queries]; used when fixed_n < 0
  float* thr;             // [n_queries] out: score of the k-th best
  int32_t cap;
  int32_t fixed_n;        // >= 0: every list has exactly this many entries
  int32_t k;
  int32_t final_pass;     // 1: write out_values / out_indices; 0: compact list + thr
  float* out_values;      // [n_queries, k]
  int64_t* out_indices;   // [n_queries, k]
  int64_t index_offset;
  int32_t* flags;
  uint64_t* out_keys;     // final pass, optional: [n_queries, k] keys with GLOBAL rows (row + index_offset)
  // segmented input (merge of all-gathered lists laid out [n_lists, n_queries, seg_len]):
  // element i of query q's list lives at cand[(i / seg_len) * seg_stride + q * seg_len + i % seg_len]
  int32_t seg_len;        // 0 = plain [n_queries, cap] layout
  int64_t seg_stride;
  // fused all-gather over NVLink peer memory (multi-GPU, see api.cu: mmrs_search_topk_fused_gather_async)
  int32_t g_role;                  // 0 none, 1 producer (last select of the local search), 2 consumer (merge)
  int32_t g_world, g_rank;
  uint64_t* const* g_peer_bufs;    // [g_world] every rank's gather buffer (peer-mapped)
  uint32_t* const* g_peer_flags;   // [g_world] every rank's flag array: [0,world) ready, [world,2*world) ack
  int64_t g_list_stride;           // elements between two ranks' lists inside a gather buffer
  int32_t g_status_index;          // element of a list that carries the rank's status word
  const uint32_t* g_epoch;         // device: sequence number of this call on this slot (starts at 1)
  uint32_t* g_counter;             // device: CTAs done (returns to 0)
  uint32_t* g_status_out;          // consumer: [g_world] private snapshot of the ranks' status words
  // row-filtered search: fewer than k non-zero keys is legitimate (few allowed rows seen so far, or a
  // shard with fewer than k allowed rows).  Non-final pass: thr = -inf, so the next phase appends every
  // allowed row; final pass: positions n_win .. k-1 get value -inf, index -1, key 0.
  int32_t pad_short;
};

// launchers called from another file than the one that defines them
// Fused all-gather bookkeeping done by block 0 of the prep kernel (the first kernel of a call):
// bump the slot's epoch and wait until every rank has acknowledged the previous one.
struct GatherPrologue {
  uint32_t* epoch;            // nullptr: not a fused-gather call
  const uint32_t* ack_flags;  // this rank's ack flags [world]
  int32_t world;
  uint64_t timeout_ns;
};
cudaError_t launch_prep_queries(const float* q, int32_t n_queries, int64_t ldq, int32_t dim,
                                int32_t normalize, int32_t round_bf16, float* out_f32,
                                __nv_bfloat16* out_bf16, int32_t n_rows_padded, int32_t ld_out,
                                int32_t* flags, const GatherPrologue& gp, cudaStream_t stream);
const void* prep_kernel_handle();     // for CUDA-graph node patching (api.cu)
constexpr int kPrepKernelParams = 12;
const void* select_kernel_handle();
cudaError_t launch_gather_wait(const uint32_t* my_flags, int32_t world, const uint32_t* epoch, int32_t* status,
                               uint64_t timeout_ns, cudaStream_t stream);
cudaError_t launch_scan_gemv(const ScanParams& p, int32_t dtype, int mode, int sm_count,
                             cudaStream_t stream);
// refine (scan_gemv.cu): one key per (query, candidate) into keys [n_queries, k_cand]
cudaError_t launch_refine_scores(const void* store, int32_t dtype, int64_t n_rows, int64_t ld, int32_t dim,
                                 const float* queries, int32_t ldq, float scale, const int64_t* cand,
                                 int32_t n_queries, int32_t k_cand, uint64_t* keys, int32_t* flags,
                                 cudaStream_t stream);
cudaError_t launch_quantize_rows_i8(const void* src, int32_t src_dtype, int64_t n_rows, int32_t dim, int64_t ld_src,
                                    int8_t* dst, int64_t ld_dst, int32_t* status, int sm_count, cudaStream_t stream);
cudaError_t launch_select(const SelectParams& p, int32_t n_queries, cudaStream_t stream);
cudaError_t launch_fill_u32(uint32_t* p, uint32_t v, int64_t n, cudaStream_t stream);
cudaError_t launch_pack_row_filter(const uint8_t* allowed, int64_t n_rows, uint32_t* words, int64_t n_words,
                                   unsigned long long* count, int sm_count, cudaStream_t stream);
cudaError_t launch_pack_keys(const float* values, const int64_t* indices, int32_t n_lists,
                             int32_t n_queries, int32_t k_in, uint64_t* cand, int32_t cap,
                             cudaStream_t stream);
// K2.  q_bf16 is the prepared [n_q_padded, ldq] bf16 query matrix; handles up to 256 queries.
// g_plane_rows: rows between two planes of a bf16x3 gallery (the full gallery's n_rows).
// i8: an int8 gallery with the prepared int8 query rows in q_bf16.
cudaError_t launch_scan_mma(const ScanParams& p, const __nv_bfloat16* q_bf16, int32_t n_q_padded,
                            int mode, int32_t* flags, int sm_count, cudaStream_t stream, int split,
                            int64_t g_plane_rows, bool i8 = false);
int scan_mma_max_queries();
int scan_mma_split_max_queries();
cudaError_t launch_split_bf16x3(const float* src, int64_t n_rows, int32_t dim, int64_t ld_src, __nv_bfloat16* dst,
                                int64_t ld_dst, int sm_count, cudaStream_t stream);
// range search finalize (range.cu)
int64_t range_chunks(int64_t n_words);
cudaError_t launch_range_mark_prefix(const uint64_t* cand, int64_t cap, const uint32_t* cnt, int32_t n_queries,
                                     uint32_t* bitmap, uint32_t* word_base, uint32_t* chunk_sum, int64_t* total,
                                     int sm_count, cudaStream_t stream);
cudaError_t launch_range_scatter(const uint64_t* cand, int64_t cap, const uint32_t* cnt, int32_t n_queries,
                                 const uint32_t* bitmap, const uint32_t* word_base, const int64_t* out_off,
                                 int64_t index_offset, float* values, int64_t* indices, int sm_count,
                                 cudaStream_t stream);
// lexicographic sort of [n_pairs, 2] row pairs (selfjoin.cu); scratch: mmrs_sort_pairs_workspace_bytes(n_pairs)
cudaError_t launch_sort_pairs(int64_t* pairs, int64_t n_pairs, uint64_t* scratch, cudaStream_t stream);

}  // namespace mmrs
