// api.cu -- the extern "C" boundary declared in include/mmrs_b200.h and the host-side
// orchestration of a search: query preparation, the phase schedule of plan.h, kernel choice
// (K1 streaming GEMV for small batches, K2 tcgen05 for the rest), the status read-back and the
// exhaustive re-run of a query whose candidate list overflowed.
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <mutex>
#include <vector>

#include "common.cuh"
#include "plan.h"

namespace mmrs {

// implemented in selfjoin.cu / scan_mma.cu
cudaError_t launch_selfjoin_f32(const float* emb, int64_t n_rows, int32_t dim, int64_t ld,
                                float threshold, int64_t row_begin, int64_t row_end,
                                int64_t* out_pairs, int64_t capacity, int64_t* out_count,
                                int sm_count, cudaStream_t stream);
cudaError_t launch_threshold_sweep(const float* pos, int64_t n_pos, const float* neg, int64_t n_neg,
                                   const double* thr, int32_t n_thr, int64_t* out_counts,
                                   unsigned long long* hist_ws, int sm_count, cudaStream_t stream);
cudaError_t launch_threshold_sweep_f64(const double* pos, int64_t n_pos, const double* neg, int64_t n_neg,
                                       const double* thr, int32_t n_thr, int64_t* out_counts,
                                       unsigned long long* hist_ws, int sm_count, cudaStream_t stream);
cudaError_t launch_sort_pairs(int64_t* pairs, int64_t n_pairs, uint64_t* scratch, cudaStream_t stream);
cudaError_t launch_threshold_sweep_labeled(const float* scores, const int64_t* targets, int64_t label, int64_t n,
                                           int32_t n_thr, int32_t grid_f32, double* thr_out, int64_t* out_counts,
                                           unsigned long long* hist_ws, uint32_t* mm_ws, int sm_count,
                                           cudaStream_t stream);
cudaError_t launch_score_range_batched(const float* scores, int64_t ld, int32_t n_q, int64_t n, const uint32_t* filt,
                                       uint32_t* range, int sm_count, cudaStream_t stream);
cudaError_t launch_threshold_sweep_batched(const float* scores, int64_t ld, int32_t n_q, int64_t n,
                                           const int32_t* row_labels, const int32_t* query_labels, const uint32_t* filt,
                                           const uint32_t* range, int32_t n_thr, int32_t grid_f32, double* thr_out,
                                           int64_t* out_counts, int64_t* out_n_pos, unsigned long long* hist_ws,
                                           int sm_count, cudaStream_t stream);
// K5 on tensor cores (selfjoin_mma.cu)
bool sjm_pair_mode(int64_t n_rows, int32_t dim, int32_t world);
int64_t sjm_plan(int64_t n_rows, int32_t rank, int32_t world, bool pair, int64_t* h_panel_start, int32_t max_panels,
                 int32_t* n_my_panels);
int64_t sjm_max_panels(int64_t n_rows);
cudaError_t launch_selfjoin_mma(const __nv_bfloat16* emb16, int64_t n_rows, int32_t dim, int64_t ld16,
                                float thr_lo, int32_t rank, int32_t world, bool pair, const int64_t* d_panel_start,
                                int32_t n_my_panels, int64_t total_tiles, int64_t* cand, int64_t cand_cap,
                                unsigned long long* cand_count, int32_t* flags, int sm_count,
                                cudaStream_t stream);
cudaError_t launch_selfjoin_recheck(const int64_t* cand, int64_t n_cand, const float* emb, int64_t ld, int32_t dim,
                                    float threshold, int64_t* out_pairs, int64_t capacity,
                                    unsigned long long* out_count, cudaStream_t stream);
// K2.  q_bf16 is the prepared [n_q_padded, ldq] bf16 query matrix; handles up to 256 queries.
// g_plane_rows: rows between two planes of a bf16x3 gallery (the full gallery's n_rows).
cudaError_t launch_scan_mma(const ScanParams& p, const __nv_bfloat16* q_bf16, int32_t n_q_padded,
                            int mode, int32_t* flags, int sm_count, cudaStream_t stream, int split,
                            int64_t g_plane_rows);
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
// greedy first-keeper resolve (dedup_resolve.cu)
cudaError_t launch_resolve_rank(const int64_t* order, int64_t n_order, int64_t n_items, uint32_t* rank, int32_t* status,
                                int sm_count, cudaStream_t stream);
cudaError_t launch_resolve_orient(const int64_t* pairs, int64_t n_pairs, int64_t n_items, const uint32_t* rank,
                                  int64_t* edges, int32_t* status, int sm_count, cudaStream_t stream);
cudaError_t launch_resolve_offsets(const int64_t* edges, int64_t n_edges, int64_t n_order, int64_t* off, int64_t* cursor,
                                   int sm_count, cudaStream_t stream);
cudaError_t launch_resolve_round(const int32_t* wl_in, const uint32_t* cnt_in, int64_t n_first, int64_t n_bound,
                                 int32_t* wl_out, uint32_t* cnt_out, const int64_t* off, const int64_t* edges,
                                 int64_t* cursor, int32_t* res, int sm_count, cudaStream_t stream);
cudaError_t launch_resolve_tail(const int32_t* wl, const uint32_t* cnt, int64_t n_bound, uint32_t* range,
                                const int64_t* off, const int64_t* edges, const int64_t* cursor, int32_t* res,
                                int sm_count, cudaStream_t stream);
cudaError_t launch_resolve_map_back(const int64_t* order, int64_t n_order, int64_t n_items, const int32_t* res,
                                    int64_t* rep, int sm_count, cudaStream_t stream);
int scan_mma_max_queries();
int scan_mma_split_max_queries();
bool scan_mma_available();

static thread_local char g_err[512] = "";

static int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

#define MMRS_CUDA(expr)                                                                     \
  do {                                                                                      \
    cudaError_t e__ = (expr);                                                               \
    if (e__ != cudaSuccess)                                                                 \
      return fail(MMRS_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__),  \
                  __FILE__, __LINE__);                                                      \
  } while (0)

// ---- measurement hooks ---------------------------------------------------------------------------
static std::atomic<long long> g_launches{0};
struct ProfRec { cudaEvent_t e0, e1; int32_t kind; int64_t bytes; int64_t flops; };
static std::mutex g_prof_mu;
static std::vector<ProfRec> g_prof;
static std::atomic<int> g_prof_on{0};

#define MMRS_LAUNCH(expr)        \
  do {                           \
    g_launches.fetch_add(1);     \
    MMRS_CUDA(expr);             \
  } while (0)

static int64_t rows_in_schedule(const TileSchedule& s, int64_t n_rows) {
  int64_t rows = 0;
  for (int64_t j = 0; j < s.n_sel; ++j) {
    const int64_t t = j * s.tile_inc;
    if (s.tile_exc != 0 && t % s.tile_exc == 0) continue;
    const int64_t r0 = t * kTileRows;
    rows += (n_rows - r0) < kTileRows ? (n_rows - r0) : kTileRows;
  }
  return rows;
}

static int env_int_early(const char* name, int dflt) {
  const char* s = getenv(name);
  return (s && *s) ? atoi(s) : dflt;
}

struct DeviceInfo {
  int device = -1;
  int sm_count = 0;
  int cc_major = 0;
};

static int current_device(DeviceInfo* info) {
  static thread_local DeviceInfo cache[64];
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess)
    return fail(MMRS_ERR_CUDA, "cudaGetDevice failed: %s (no CUDA device? this library has no CPU path)",
                cudaGetErrorString(e));
  if (dev < 0 || dev >= 64) return fail(MMRS_ERR_ARG, "device ordinal %d out of range", dev);
  if (cache[dev].device != dev) {
    DeviceInfo d;
    d.device = dev;
    MMRS_CUDA(cudaDeviceGetAttribute(&d.cc_major, cudaDevAttrComputeCapabilityMajor, dev));
    MMRS_CUDA(cudaDeviceGetAttribute(&d.sm_count, cudaDevAttrMultiProcessorCount, dev));
    cache[dev] = d;
  }
  *info = cache[dev];
  if (info->cc_major != 10)
    return fail(MMRS_ERR_ARCH, "device %d is compute capability %d.x; this library is sm_100a only",
                dev, info->cc_major);
  return MMRS_OK;
}

bool pdl_enabled() {
  static const bool on = env_int_early("MMRS_NO_PDL", 0) == 0;
  return on;
}


static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

static int env_int(const char* name, int dflt) {
  const char* s = getenv(name);
  if (!s || !*s) return dflt;
  return atoi(s);
}

constexpr int kSuperChunk = 1024;  // queries sharing one set of candidate lists

// Every phase appends about k * ratio keys per query whatever its size, so the appends of a whole
// search scale with n_queries * k * ratio * (#phases - 1): small batches take few, coarse phases
// (launch-bound), large batches finer ones (append-bound).  Measured on B200: tools/tune_plan.sh.
static SearchPlan plan_for(int64_t n_rows, int32_t k, int32_t n_queries) {
  // profiles/r01_tune4.log: seed sample of 32-64 tiles, a mid phase 8x as large, everything else last
  const int ratio_dflt = 3;
  // 40-48 queries: 0.193 ms per step with 64 seed tiles against 0.200-0.209 with 32; no difference up to 32
  const int dense_dflt = n_queries <= 32 ? 32 : 64;
  return make_search_plan(n_rows, k, kTileRows, env_int("MMRS_RATIO_LOG2", ratio_dflt),
                          env_int("MMRS_DENSE_TILES", dense_dflt));
}

static int32_t padded_dim(int32_t dim) { return (dim + 7) / 8 * 8; }
static int32_t padded_queries(int32_t nq) { return (nq + 15) / 16 * 16; }

struct Workspace {
  int32_t* flags;          // [8]
  float* q_f32;            // [Qp, ldq]
  __nv_bfloat16* q_bf16;   // [Qp, ldq]
  float* thr;              // [Qs]
  uint32_t* cnt;           // [Qs]
  uint64_t* cand;          // [Qs, cap] (>= n_tiles * kTileRows keys for the exhaustive path)
  size_t cand_keys;
  uint32_t* gscratch;      // [kGScratch] fused all-gather bookkeeping, see below
  size_t total;
};
// gscratch words: [0] epoch of the slot (bumped by the prep kernel of every fused call; the caller
// zero-fills a workspace once, before its first use) [1] producer CTA counter [2] consumer CTA counter
// [8, 8 + world) snapshot of the ranks' status words [8 + world] status of the merge select
constexpr int kGScratch = 128;
constexpr int kGStatus = 8;
constexpr int kMaxWorld = 64;

static Workspace carve(void* base, int64_t n_rows, int32_t dim, int32_t n_queries, int32_t k,
                       bool with_lists, bool exhaustive = false) {
  Workspace w{};
  size_t off = 0;
  char* b = static_cast<char*>(base);
  auto take = [&](size_t bytes) { char* p = b ? b + off : nullptr; off += align_up(bytes, 256); return p; };
  const int32_t ldq = padded_dim(dim), qp = padded_queries(n_queries);
  w.flags = reinterpret_cast<int32_t*>(take(8 * sizeof(int32_t)));
  w.gscratch = reinterpret_cast<uint32_t*>(take(kGScratch * sizeof(uint32_t)));
  w.q_f32 = reinterpret_cast<float*>(take(static_cast<size_t>(qp) * ldq * sizeof(float)));
  w.q_bf16 = reinterpret_cast<__nv_bfloat16*>(take(3 * static_cast<size_t>(qp) * ldq * sizeof(__nv_bfloat16)));   // up to 3 planes
  if (with_lists) {
    const SearchPlan pl = plan_for(n_rows, k, n_queries);
    const int32_t qs = n_queries < kSuperChunk ? n_queries : kSuperChunk;
    w.thr = reinterpret_cast<float*>(take(static_cast<size_t>(qs) * sizeof(float)));
    w.cnt = reinterpret_cast<uint32_t*>(take(static_cast<size_t>(qs) * sizeof(uint32_t)));
    // the exhaustive re-run (one query at a time, every row a key) needs n_tiles * 128 keys -- 0.8 GB
    // at 100M rows -- and is carved only for mmrs_search_topk_exhaustive's own, temporary workspace
    size_t keys = exhaustive ? static_cast<size_t>(pl.n_tiles) * kTileRows : static_cast<size_t>(qs) * pl.cap;
    w.cand_keys = keys;
    w.cand = reinterpret_cast<uint64_t*>(take(keys * sizeof(uint64_t)));
  }
  w.total = off;
  return w;
}

// Range search (mmrs_range_search_window / _scatter): the query matrices of carve() plus, per query, a
// candidate list of one window (cap = window_rows keys), its counter, the window's row bitmap, the word
// prefix sums, the chunk sums of the prefix and the total.
// K2 stages its queries in UMMA columns padded up to 256 per launch; a padded column's threshold is +inf and
// its query row zero, so only a NaN score (a NaN or infinite gallery value times 0) passes it, and K2 appends
// that row to list q0 + column >= n_queries.  Those counters exist here and start at the list capacity, so
// the kernel's `pos < cap` test drops the appends: no key memory is needed for the padded lists.
constexpr int kRangePadLists = 256;

struct RangeWorkspace {
  Workspace base;          // flags, q_f32, q_bf16
  uint32_t* cnt;           // [Q + kRangePadLists]
  uint64_t* cand;          // [Q, window_rows]
  uint32_t* bitmap;        // [Q, window_rows / 32]
  uint32_t* word_base;     // [Q, window_rows / 32]
  uint32_t* chunk_sum;     // [Q, range_chunks(window_rows / 32)]
  int64_t* total;          // [Q]
  size_t total_bytes;
};

static RangeWorkspace carve_range(void* base, int64_t window_rows, int32_t dim, int32_t n_queries) {
  RangeWorkspace r{};
  r.base = carve(base, window_rows, dim, n_queries, 1, false);
  size_t off = r.base.total;
  char* b = static_cast<char*>(base);
  auto take = [&](size_t bytes) { char* p = b ? b + off : nullptr; off += align_up(bytes, 256); return p; };
  const size_t q = static_cast<size_t>(n_queries), words = static_cast<size_t>(window_rows / 32);
  r.cnt = reinterpret_cast<uint32_t*>(take((q + kRangePadLists) * sizeof(uint32_t)));
  r.cand = reinterpret_cast<uint64_t*>(take(q * static_cast<size_t>(window_rows) * sizeof(uint64_t)));
  r.bitmap = reinterpret_cast<uint32_t*>(take(q * words * sizeof(uint32_t)));
  r.word_base = reinterpret_cast<uint32_t*>(take(q * words * sizeof(uint32_t)));
  r.chunk_sum = reinterpret_cast<uint32_t*>(take(q * static_cast<size_t>(range_chunks(window_rows / 32)) * sizeof(uint32_t)));
  r.total = reinterpret_cast<int64_t*>(take(q * sizeof(int64_t)));
  r.total_bytes = off;
  return r;
}

// Duplicate resolve (mmrs_resolve_duplicates): a 256-byte header, then the rank, edge, CSR, decision and
// worklist arrays of dedup_resolve.cu.
struct ResolveWorkspace {
  int32_t* header;         // [0] status bits, [1] [2] worklist counters, [4] [5] worklist rank range
  uint32_t* rank;          // [n_items] rank of each row, 0xffffffff = not in the order
  int64_t* edges;          // [n_pairs, 2] oriented (high rank, low rank), sorted in place
  uint64_t* sort;          // mmrs_sort_pairs_workspace_bytes(n_pairs)
  int64_t* off;            // [n_order + 1] first edge of each rank
  int64_t* cursor;         // [n_order] next edge each undecided rank looks at
  int32_t* res;            // [n_order] -1 undecided, r kept, else the representative's rank
  int32_t* wl[2];          // [n_order] each: worklists of undecided ranks, ping-pong
  size_t total_bytes;
};

static ResolveWorkspace carve_resolve(void* base, int64_t n_items, int64_t n_order, int64_t n_pairs) {
  ResolveWorkspace r{};
  size_t off = 0;
  char* b = static_cast<char*>(base);
  auto take = [&](size_t bytes) { char* p = b ? b + off : nullptr; off += align_up(bytes, 256); return p; };
  const size_t items = static_cast<size_t>(n_items), ord = static_cast<size_t>(n_order),
               pairs = static_cast<size_t>(n_pairs);
  r.header = reinterpret_cast<int32_t*>(take(256));
  r.rank = reinterpret_cast<uint32_t*>(take(items * sizeof(uint32_t)));
  r.edges = reinterpret_cast<int64_t*>(take(pairs * 2 * sizeof(int64_t)));
  r.sort = reinterpret_cast<uint64_t*>(take(mmrs_sort_pairs_workspace_bytes(n_pairs)));
  r.off = reinterpret_cast<int64_t*>(take((ord + 1) * sizeof(int64_t)));
  r.cursor = reinterpret_cast<int64_t*>(take(ord * sizeof(int64_t)));
  r.res = reinterpret_cast<int32_t*>(take(ord * sizeof(int32_t)));
  r.wl[0] = reinterpret_cast<int32_t*>(take(ord * sizeof(int32_t)));
  r.wl[1] = reinterpret_cast<int32_t*>(take(ord * sizeof(int32_t)));
  r.total_bytes = off;
  return r;
}
// The host reads the worklist count once per batch of rounds.  A batch that decides fewer than
// kResolveTailBelow rows per round hands the rest to the one-warp tail: a round costs a launch and a pass
// over the whole worklist, and that little progress means long dependent chains (a path in walk order
// decides about one rank per round), which the tail walks in one ascending sweep.
constexpr int kResolveBatch = 4;
constexpr int64_t kResolveTailBelow = 2048;

static int check_matrix(const void* p, int64_t n_rows, int32_t dim, int64_t ld, int32_t dtype,
                        const char* what) {
  if (!p) return fail(MMRS_ERR_ARG, "%s pointer is null", what);
  if (n_rows < 1) return fail(MMRS_ERR_ARG, "%s has %lld rows", what, (long long)n_rows);
  if (n_rows > 0xffffffffll) return fail(MMRS_ERR_ARG, "%s: more than 2^32 rows per shard", what);
  if (dtype != MMRS_DTYPE_F32 && dtype != MMRS_DTYPE_BF16 && dtype != MMRS_DTYPE_BF16X3)
    return fail(MMRS_ERR_ARG, "%s dtype %d unknown", what, dtype);
  const int elems16 = dtype == MMRS_DTYPE_F32 ? 4 : 8;
  if (dim < 1 || dim % elems16 != 0)
    return fail(MMRS_ERR_ARG, "%s dim %d must be a positive multiple of %d (pad with zeros)", what,
                dim, elems16);
  if (ld < dim || ld % elems16 != 0)
    return fail(MMRS_ERR_ARG, "%s row stride %lld must be >= dim and a multiple of %d", what,
                (long long)ld, elems16);
  if (reinterpret_cast<uintptr_t>(p) % 16 != 0)
    return fail(MMRS_ERR_ARG, "%s pointer must be 16-byte aligned", what);
  return MMRS_OK;
}

static int32_t* pinned_status() {
  static thread_local int32_t* h = nullptr;
  if (!h) {
    if (cudaHostAlloc(reinterpret_cast<void**>(&h), 8 * sizeof(int32_t), cudaHostAllocDefault) != cudaSuccess)
      h = nullptr;
  }
  return h;
}

enum class Path { kGemv, kMma };

static Path choose_path(int32_t requested, int32_t dtype, int32_t n_queries) {
  if (dtype == MMRS_DTYPE_BF16X3) return Path::kMma;   // split planes exist for the tensor cores only
  if (requested == MMRS_PATH_GEMV) return Path::kGemv;
  if (requested == MMRS_PATH_MMA) return Path::kMma;
  // measured on B200 (profiles/r01_tune3.log): K1 wins for 1-2 queries, K2 from 3 on
  if (dtype == MMRS_DTYPE_BF16 && n_queries > 2 && scan_mma_available()) return Path::kMma;
  return Path::kGemv;
}

template <typename F>
static int profiled_launch(int32_t kind, int64_t bytes, int64_t flops, cudaStream_t stream, F launch) {
  g_launches.fetch_add(1);
  if (!g_prof_on.load(std::memory_order_relaxed)) {
    MMRS_CUDA(launch());
    return MMRS_OK;
  }
  ProfRec r{};
  r.kind = kind; r.bytes = bytes; r.flops = flops;
  MMRS_CUDA(cudaEventCreate(&r.e0));
  MMRS_CUDA(cudaEventCreate(&r.e1));
  MMRS_CUDA(cudaEventRecord(r.e0, stream));
  MMRS_CUDA(launch());
  MMRS_CUDA(cudaEventRecord(r.e1, stream));
  std::lock_guard<std::mutex> lk(g_prof_mu);
  g_prof.push_back(r);
  return MMRS_OK;
}

template <typename F>
static int profiled_scan(int32_t kind, int32_t dtype, const ScanParams& p, cudaStream_t stream, F launch) {
  const int64_t rows = g_prof_on.load(std::memory_order_relaxed) ? rows_in_schedule(p.sched, p.n_rows) : 0;
  return profiled_launch(kind, rows * p.dim * (dtype == MMRS_DTYPE_BF16 ? 2 : (dtype == MMRS_DTYPE_BF16X3 ? 6 : 4)), 2 * rows * p.dim * p.nq,
                         stream, launch);
}

// One scan over the tiles of `sched` for queries [q_lo, q_hi) of the prepared matrices.
// plane_rows: rows between two bf16x3 planes when base.gallery is a row window (0: base.n_rows).
static int run_scan(Path path, const DeviceInfo& dev, int32_t dtype, ScanParams base,
                    const Workspace& w, int32_t n_q_padded, int32_t q_lo, int32_t q_hi, int mode,
                    cudaStream_t stream, int64_t plane_rows = 0) {
  if (plane_rows == 0) plane_rows = base.n_rows;
  if (path == Path::kMma) {
    // 256 queries per CTA (the UMMA N limit); when at least two full chunks remain, one launch takes
    // up to four of them and their CTAs share every gallery tile through L2 (scan_mma.cu, gridDim.y):
    // +7 % on the 64K-query C5 shard, +8 % at 1024 queries on C2
    const int split = dtype == MMRS_DTYPE_BF16X3 ? 3 : 1;
    const int wide = scan_mma_max_queries();
    for (int32_t q = q_lo; q < q_hi;) {
      const int32_t rem = q_hi - q;
      int32_t chunk = rem < 256 ? rem : 256;
      if (rem >= 512) chunk = (rem / 256 < wide / 256 ? rem / 256 : wide / 256) * 256;   // 2..4 full chunks
      if (split == 3) chunk = rem < scan_mma_split_max_queries() ? rem : scan_mma_split_max_queries();
      ScanParams p = base;
      p.q0 = q;
      p.nq = chunk;
      q += chunk;
      int rc = profiled_scan(MMRS_PATH_MMA, dtype, p, stream, [&]() {
        return launch_scan_mma(p, w.q_bf16, n_q_padded, mode, w.flags, dev.sm_count, stream, split, plane_rows);
      });
      if (rc != MMRS_OK) return rc;
    }
    return MMRS_OK;
  }
  const int chunk = dtype == MMRS_DTYPE_F32 ? 8 : 4;
  for (int32_t q = q_lo; q < q_hi; q += chunk) {
    ScanParams p = base;
    p.q0 = q;
    p.nq = (q_hi - q) < chunk ? (q_hi - q) : chunk;
    int rc = profiled_scan(MMRS_PATH_GEMV, dtype, p, stream, [&]() {
      return launch_scan_gemv(p, dtype, mode, dev.sm_count, stream);
    });
    if (rc != MMRS_OK) return rc;
  }
  return MMRS_OK;
}

static TileSchedule sched_of(const SearchPlan& pl, int i) {
  TileSchedule s;
  s.n_tiles = pl.n_tiles;
  s.tile_inc = pl.phase[i].inc;
  s.tile_exc = pl.phase[i].exc;
  s.n_sel = pl.phase[i].n_sel;
  return s;
}

struct SearchArgs {
  const void* gallery; int64_t n_rows; int32_t dim; int64_t ld; int32_t dtype;
  const float* d_queries; int32_t n_queries; int64_t ldq_in;
  int32_t k; int32_t normalize; float scale; int64_t index_offset; int32_t path;
  float* d_values; int64_t* d_indices;
  uint64_t* d_keys = nullptr;   // optional: packed (score, ~global row) keys instead of / besides the pair
  // fused all-gather: the last local select stores into every rank's gather buffer (producer), a
  // one-warp kernel waits for every rank's keys, a merge select over this rank's buffer (consumer)
  // writes d_values / d_indices [n_queries, g_k_out]
  int32_t g_world = 0, g_rank = 0;
  uint64_t* const* g_peer_bufs = nullptr;
  uint32_t* const* g_peer_flags = nullptr;
  uint64_t* g_local_buf = nullptr;
  uint32_t* g_local_flags = nullptr;
  int64_t g_list_stride = 0;
  int32_t g_k_out = 0;
  uint64_t g_timeout_ns = 0;
  const uint32_t* row_filter = nullptr;   // allow-list bitmap over the local rows (mmrs_pack_row_filter); nullptr = all
  // label-conditioned search (ScanParams): row labels over the local rows (nullptr = unlabeled), device
  // query labels [n_queries], MMRS_LABEL_SAME / MMRS_LABEL_OTHER
  const int32_t* row_labels = nullptr;
  const int32_t* query_labels = nullptr;
  int32_t label_match = 0;
  // a query may legitimately see fewer than k eligible rows: the selects pad instead of flagging
  bool pad_short() const { return row_filter != nullptr || row_labels != nullptr; }
};

static void set_labels(ScanParams& p, const SearchArgs& a) {
  p.row_labels = a.row_labels;
  p.query_labels = a.row_labels ? a.query_labels : nullptr;
  p.label_match = a.row_labels ? a.label_match : 0;
}

static uint64_t gather_timeout_ns() {
  const int ms = env_int("MMRS_GATHER_TIMEOUT_MS", 20000);
  return static_cast<uint64_t>(ms < 1 ? 1 : ms) * 1000000ull;
}

static int enqueue_prep(const SearchArgs& a, const Workspace& w, cudaStream_t stream) {
  const int32_t ldq = padded_dim(a.dim), qp = padded_queries(a.n_queries);
  GatherPrologue gp{};
  if (a.g_world > 0) {
    gp.epoch = w.gscratch; gp.ack_flags = a.g_local_flags + a.g_world; gp.world = a.g_world;
    gp.timeout_ns = a.g_timeout_ns;
  }
  return profiled_launch(4, 0, 0, stream, [&]() {
    return launch_prep_queries(a.d_queries, a.n_queries, a.ldq_in, a.dim, a.normalize,
                               a.dtype == MMRS_DTYPE_BF16 ? 1 : (a.dtype == MMRS_DTYPE_BF16X3 ? 2 : 0), w.q_f32, w.q_bf16, qp, ldq,
                               w.flags, gp, stream);
  });
}

// Enqueue the whole fused search on `stream`.  Results are valid iff the flag word stays 0.
static int enqueue_search(const SearchArgs& a, const DeviceInfo& dev, const Workspace& w,
                          cudaStream_t stream) {
  const SearchPlan pl = plan_for(a.n_rows, a.k, a.n_queries);
  const int32_t ldq = padded_dim(a.dim), qp = padded_queries(a.n_queries);
  const Path path = choose_path(a.path, a.dtype, a.n_queries);
  if (path == Path::kMma && a.dtype == MMRS_DTYPE_F32)
    return fail(MMRS_ERR_ARG, "MMRS_PATH_MMA needs a bf16 (or bf16x3) gallery");
  const bool fused = a.g_world > 0;

  MMRS_CUDA(cudaMemsetAsync(w.flags, 0, 8 * sizeof(int32_t), stream));
  if (fused)   // status snapshot + merge status of this call (the epoch and the CTA counters persist)
    MMRS_CUDA(cudaMemsetAsync(w.gscratch + kGStatus, 0, (kMaxWorld + 1) * sizeof(uint32_t), stream));
  {
    int rc = enqueue_prep(a, w, stream);
    if (rc != MMRS_OK) return rc;
  }
  ScanParams base{};
  base.gallery = a.gallery; base.n_rows = a.n_rows; base.ld = a.ld; base.dim = a.dim;
  base.queries = w.q_f32; base.ldq = ldq; base.scale = a.scale;
  base.cap = pl.cap;
  base.row_filter = a.row_filter;
  set_labels(base, a);

  for (int32_t s0 = 0; s0 < a.n_queries; s0 += kSuperChunk) {
    const int32_t s1 = (a.n_queries - s0) < kSuperChunk ? a.n_queries : s0 + kSuperChunk;
    const int32_t ns = s1 - s0;
    // list q of this super-chunk lives at cand[(q - s0) * cap]: bias the pointers so kernels
    // can index by absolute query id
    base.cand = w.cand - static_cast<int64_t>(s0) * pl.cap;
    base.cnt = w.cnt - s0;
    base.thr = w.thr - s0;
    for (int ph = 0; ph < pl.n_phases; ++ph) {
      base.sched = sched_of(pl, ph);
      const int mode = ph == 0 ? kModeDense : kModeFilter;
      int rc = run_scan(path, dev, a.dtype, base, w, qp, s0, s1, mode, stream);
      if (rc != MMRS_OK) return rc;
      SelectParams sp{};
      sp.cand = w.cand; sp.cnt = w.cnt; sp.thr = w.thr; sp.cap = pl.cap;
      sp.fixed_n = ph == 0 ? pl.dense_rows : -1;
      sp.k = a.k;
      sp.final_pass = ph == pl.n_phases - 1;
      if (!fused) {
        sp.out_values = a.d_values ? a.d_values + static_cast<int64_t>(s0) * a.k : nullptr;
        sp.out_indices = a.d_indices ? a.d_indices + static_cast<int64_t>(s0) * a.k : nullptr;
        sp.out_keys = a.d_keys ? a.d_keys + static_cast<int64_t>(s0) * a.k : nullptr;
      }
      sp.index_offset = a.index_offset;
      sp.flags = w.flags;
      sp.pad_short = a.pad_short();
      if (fused && sp.final_pass) {
        sp.g_role = 1; sp.g_world = a.g_world; sp.g_rank = a.g_rank;
        sp.g_peer_bufs = a.g_peer_bufs; sp.g_peer_flags = a.g_peer_flags;
        sp.g_list_stride = a.g_list_stride; sp.g_status_index = a.n_queries * a.k;
        sp.g_epoch = w.gscratch; sp.g_counter = w.gscratch + 1;
      }
      rc = profiled_launch(3, 0, 0, stream, [&]() { return launch_select(sp, ns, stream); });
      if (rc != MMRS_OK) return rc;
    }
  }
  if (fused) {
    int32_t* merge_status = reinterpret_cast<int32_t*>(w.gscratch + kGStatus + a.g_world);
    int rc = profiled_launch(5, 0, 0, stream, [&]() {
      return launch_gather_wait(a.g_local_flags, a.g_world, w.gscratch, merge_status, a.g_timeout_ns, stream);
    });
    if (rc != MMRS_OK) return rc;
    // consumer: merge the lists every rank stored into MY gather buffer
    SelectParams sp{};
    sp.cand = a.g_local_buf;
    sp.cap = a.g_world * a.k; sp.fixed_n = a.g_world * a.k; sp.k = a.g_k_out; sp.final_pass = 1;
    sp.out_values = a.d_values; sp.out_indices = a.d_indices; sp.index_offset = 0;
    sp.flags = merge_status;
    sp.seg_len = a.k; sp.seg_stride = a.g_list_stride;
    sp.g_role = 2; sp.g_world = a.g_world; sp.g_rank = a.g_rank; sp.g_peer_bufs = a.g_peer_bufs; sp.g_peer_flags = a.g_peer_flags;
    sp.g_list_stride = a.g_list_stride; sp.g_status_index = a.n_queries * a.k;
    sp.g_epoch = w.gscratch; sp.g_counter = w.gscratch + 2; sp.g_status_out = w.gscratch + kGStatus;
    sp.pad_short = a.pad_short();
    rc = profiled_launch(3, 0, 0, stream, [&]() { return launch_select(sp, a.n_queries, stream); });
    if (rc != MMRS_OK) return rc;
  }
  return MMRS_OK;
}

// Slow exact path for when a candidate list overflowed: one query at a time, every score
// becomes a key, one select over all of them.  `w` is carved with exhaustive = true.
static int enqueue_exhaustive(const SearchArgs& a, const DeviceInfo& dev, const Workspace& w,
                              cudaStream_t stream) {
  const SearchPlan pl = plan_for(a.n_rows, a.k, a.n_queries);
  const int32_t ldq = padded_dim(a.dim);
  const int32_t all_rows = pl.n_tiles * kTileRows;
  ScanParams base{};
  base.gallery = a.gallery; base.n_rows = a.n_rows; base.ld = a.ld; base.dim = a.dim;
  base.queries = w.q_f32; base.ldq = ldq; base.scale = a.scale;
  base.cap = all_rows;
  base.sched = TileSchedule{pl.n_tiles, 1, 0, pl.n_tiles};
  base.row_filter = a.row_filter;
  set_labels(base, a);   // one query per pass below, with that query's own label (query_labels[q0])
  MMRS_CUDA(cudaMemsetAsync(w.flags, 0, 8 * sizeof(int32_t), stream));
  {
    int rc = enqueue_prep(a, w, stream);
    if (rc != MMRS_OK) return rc;
  }
  for (int32_t q = 0; q < a.n_queries; ++q) {
    ScanParams p = base;
    p.cand = w.cand - static_cast<int64_t>(q) * all_rows;
    p.q0 = q; p.nq = 1;
    if (a.dtype == MMRS_DTYPE_BF16X3) {
      MMRS_LAUNCH(launch_scan_mma(p, w.q_bf16, padded_queries(a.n_queries), kModeDense, w.flags, dev.sm_count, stream, 3,
                                   a.n_rows));
    } else {
      MMRS_LAUNCH(launch_scan_gemv(p, a.dtype, kModeDense, dev.sm_count, stream));
    }
    SelectParams sp{};
    sp.cand = w.cand; sp.cnt = w.cnt; sp.thr = w.thr; sp.cap = all_rows;
    sp.fixed_n = all_rows; sp.k = a.k; sp.final_pass = 1;
    sp.out_values = a.d_values + static_cast<int64_t>(q) * a.k;
    sp.out_indices = a.d_indices + static_cast<int64_t>(q) * a.k;
    sp.index_offset = a.index_offset; sp.flags = w.flags;
    sp.pad_short = a.pad_short();
    MMRS_LAUNCH(launch_select(sp, 1, stream));
  }
  return MMRS_OK;
}

// ---- CUDA-graph cache -----------------------------------------------------------------------------
// A search is 7-9 short dependent launches in front of one long one; submitted one by one the GPU
// idles between them (the host needs ~60 us to issue what the GPU runs in ~40 us, measured:
// profiles/r01_v1_bench.json whole step 0.31 ms vs 0.24 ms of kernels).  The whole sequence
// is therefore captured once per workspace slot and call signature and replayed with one
// cudaGraphLaunch.  The key is the WORKSPACE (one per search shape and stream) plus everything that
// shapes the launches; the caller's query and result pointers are NOT part of it: they appear in
// exactly two kinds of kernel node -- the prep kernel reads d_queries, the final select(s) write
// d_values / d_indices / d_keys -- and those nodes are re-pointed with
// cudaGraphExecKernelNodeSetParams when a call brings other tensors.  A caller that keeps every result
// tensor therefore still replays one graph (tests/test_search_gpu.py::test_retained_outputs_capture_once).
struct GraphKey {
  const void* gallery; int64_t n_rows; int32_t dim; int64_t ld; int32_t dtype;
  int32_t n_queries; int64_t ldq_in; int32_t k; int32_t normalize;
  float scale; int64_t index_offset; int32_t path;
  void* workspace; int device; int ratio_log2; int dense_tiles;
  bool has_values, has_indices, has_keys;
  int32_t g_world, g_rank; const void* g_bufs; const void* g_flags; const void* g_local_buf; const void* g_local_flags;
  int64_t g_stride; int32_t g_k_out; uint64_t g_timeout_ns;
  uint64_t knobs;   // the kernel-shape environment knobs the captured launches were configured with
  const void* row_filter;   // the captured scans read the bitmap through this pointer
  const void* row_labels; const void* query_labels; int32_t label_match;   // and the labels through these
  bool operator==(const GraphKey& o) const {
    return knobs == o.knobs && row_filter == o.row_filter && row_labels == o.row_labels &&
           query_labels == o.query_labels && label_match == o.label_match && g_world == o.g_world && g_rank == o.g_rank && g_bufs == o.g_bufs && g_flags == o.g_flags &&
           g_local_buf == o.g_local_buf && g_local_flags == o.g_local_flags && g_stride == o.g_stride && g_k_out == o.g_k_out &&
           g_timeout_ns == o.g_timeout_ns && has_values == o.has_values && has_indices == o.has_indices &&
           has_keys == o.has_keys && gallery == o.gallery && n_rows == o.n_rows && dim == o.dim && ld == o.ld &&
           dtype == o.dtype && n_queries == o.n_queries && ldq_in == o.ldq_in && k == o.k &&
           normalize == o.normalize && scale == o.scale && index_offset == o.index_offset &&
           path == o.path && workspace == o.workspace && device == o.device && ratio_log2 == o.ratio_log2 &&
           dense_tiles == o.dense_tiles;
  }
};
// FNV-1a over the values of the MMRS_K2_* / MMRS_NO_PDL knobs (read per launch by the kernels' host
// side): a graph captured under one setting must not be replayed under another
static uint64_t knob_hash() {
  static const char* const kNames[] = {"MMRS_K2_SMALL_MAX", "MMRS_K2_BIG_SMEM", "MMRS_K2_CTAS_PER_SM", "MMRS_K2_QCHUNKS",
                                       "MMRS_K2_NO_PAIR", "MMRS_K2_PAIR_MIN", "MMRS_K2_DEBUG_SKIP_EPI", "MMRS_NO_PDL",
                                       "MMRS_K2_STICKY", "MMRS_K2_HBM_PAIRS", "MMRS_K2_PREFETCH", "MMRS_K2_SMALL_PAIR_MAX"};
  uint64_t h = 1469598103934665603ull;
  for (const char* name : kNames) {
    const char* v = getenv(name);
    for (const char* c = v ? v : "\x01"; *c; ++c) h = (h ^ static_cast<unsigned char>(*c)) * 1099511628211ull;
    h = (h ^ 0xffu) * 1099511628211ull;
  }
  return h;
}
enum SiteKind { kSitePrep = 0, kSiteFinalSelect = 1 };
struct PatchSite { cudaGraphNode_t node; int kind; int64_t s0; };
struct GraphEntry {
  GraphKey key; cudaGraph_t graph; cudaGraphExec_t exec; uint64_t stamp; long long kernels;
  std::vector<PatchSite> sites; bool patchable;
  const float* q; float* v; int64_t* i; uint64_t* keys;   // the pointers the executable graph currently holds
};
static std::mutex g_graph_mu;
static std::vector<GraphEntry> g_graphs;
static uint64_t g_graph_clock = 0;
constexpr size_t kMaxGraphs = 32;
static std::atomic<long long> g_stat_captures{0}, g_stat_replays{0}, g_stat_patches{0}, g_stat_unpatchable{0};

// Find the kernel nodes that hold caller pointers.  False when the graph does not look as expected
// (then the entry only serves calls with exactly the captured pointers).
static bool discover_sites(cudaGraph_t graph, const SearchArgs& a, std::vector<PatchSite>* sites) {
  size_t n = 0;
  if (cudaGraphGetNodes(graph, nullptr, &n) != cudaSuccess || n == 0) { cudaGetLastError(); return false; }
  std::vector<cudaGraphNode_t> nodes(n);
  if (cudaGraphGetNodes(graph, nodes.data(), &n) != cudaSuccess) { cudaGetLastError(); return false; }
  const int32_t k_out = a.g_world > 0 ? a.g_k_out : a.k;
  int n_prep = 0, n_final = 0;
  for (cudaGraphNode_t node : nodes) {
    cudaGraphNodeType t;
    if (cudaGraphNodeGetType(node, &t) != cudaSuccess) { cudaGetLastError(); return false; }
    if (t != cudaGraphNodeTypeKernel) continue;
    cudaKernelNodeParams kp{};
    if (cudaGraphKernelNodeGetParams(node, &kp) != cudaSuccess) { cudaGetLastError(); return false; }
    if (kp.func == prep_kernel_handle()) {
      if (!kp.kernelParams || *static_cast<const float* const*>(kp.kernelParams[0]) != a.d_queries) return false;
      sites->push_back(PatchSite{node, kSitePrep, 0});
      ++n_prep;
    } else if (kp.func == select_kernel_handle()) {
      if (!kp.kernelParams) return false;
      const SelectParams* sp = static_cast<const SelectParams*>(kp.kernelParams[0]);
      if (!sp->final_pass || (a.g_world > 0 && sp->g_role != 2)) continue;
      int64_t off = -1;
      if (a.d_values && sp->out_values) off = sp->out_values - a.d_values;
      else if (a.d_indices && sp->out_indices) off = sp->out_indices - a.d_indices;
      else if (a.d_keys && sp->out_keys) off = static_cast<int64_t>(sp->out_keys - a.d_keys);
      if (off < 0 || off % k_out != 0) return false;
      sites->push_back(PatchSite{node, kSiteFinalSelect, off / k_out});
      ++n_final;
    }
  }
  const int want_final = a.g_world > 0 ? 1 : (a.n_queries + kSuperChunk - 1) / kSuperChunk;
  return n_prep == 1 && n_final == want_final;
}

static int patch_entry(GraphEntry& e, const SearchArgs& a) {
  const int32_t k_out = a.g_world > 0 ? a.g_k_out : a.k;
  for (const PatchSite& site : e.sites) {
    cudaKernelNodeParams kp{};
    MMRS_CUDA(cudaGraphKernelNodeGetParams(site.node, &kp));
    void* params[kPrepKernelParams];
    if (site.kind == kSitePrep) {
      for (int i = 0; i < kPrepKernelParams; ++i) params[i] = kp.kernelParams[i];
      const float* q = a.d_queries;
      params[0] = &q;
      kp.kernelParams = params;
      MMRS_CUDA(cudaGraphExecKernelNodeSetParams(e.exec, site.node, &kp));
    } else {
      SelectParams sp = *static_cast<const SelectParams*>(kp.kernelParams[0]);
      sp.out_values = a.d_values ? a.d_values + site.s0 * k_out : nullptr;
      sp.out_indices = a.d_indices ? a.d_indices + site.s0 * k_out : nullptr;
      if (a.g_world == 0) sp.out_keys = a.d_keys ? a.d_keys + site.s0 * k_out : nullptr;
      params[0] = &sp;
      kp.kernelParams = params;
      MMRS_CUDA(cudaGraphExecKernelNodeSetParams(e.exec, site.node, &kp));
    }
  }
  e.q = a.d_queries; e.v = a.d_values; e.i = a.d_indices; e.keys = a.d_keys;
  g_stat_patches.fetch_add(1);
  return MMRS_OK;
}

static int launch_search_graph(const SearchArgs& a, const DeviceInfo& dev, const Workspace& w,
                               void* workspace, cudaStream_t stream) {
  if (g_prof_on.load(std::memory_order_relaxed) || env_int("MMRS_NO_GRAPH", 0))
    return enqueue_search(a, dev, w, stream);   // event-bracketed launches are issued directly
  GraphKey key{a.gallery, a.n_rows, a.dim, a.ld, a.dtype, a.n_queries, a.ldq_in, a.k,
               a.normalize, a.scale, a.index_offset, a.path, workspace,
               dev.device, env_int("MMRS_RATIO_LOG2", -1), env_int("MMRS_DENSE_TILES", -1),
               a.d_values != nullptr, a.d_indices != nullptr, a.d_keys != nullptr,
               a.g_world, a.g_rank, a.g_peer_bufs, a.g_peer_flags, a.g_local_buf, a.g_local_flags, a.g_list_stride,
               a.g_k_out, a.g_timeout_ns, knob_hash(), a.row_filter,
               a.row_labels, a.row_labels ? a.query_labels : nullptr, a.row_labels ? a.label_match : 0};
  // the lock is held across patch + launch: an executable graph must not be updated or launched from
  // two threads at once (two threads sharing one workspace would be a caller bug anyway)
  std::lock_guard<std::mutex> lk(g_graph_mu);
  GraphEntry* hit = nullptr;
  for (GraphEntry& e : g_graphs) {
    if (!(e.key == key)) continue;
    const bool same = e.q == a.d_queries && e.v == a.d_values && e.i == a.d_indices && e.keys == a.d_keys;
    if (same || e.patchable) { hit = &e; break; }
  }
  if (hit) {
    hit->stamp = ++g_graph_clock;
    if (!(hit->q == a.d_queries && hit->v == a.d_values && hit->i == a.d_indices && hit->keys == a.d_keys)) {
      int rc = patch_entry(*hit, a);
      if (rc != MMRS_OK) return rc;
    }
    g_launches.fetch_add(hit->kernels);   // a replay launches the same kernels the capture recorded
    g_stat_replays.fetch_add(1);
    MMRS_CUDA(cudaGraphLaunch(hit->exec, stream));
    return MMRS_OK;
  }
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t exec = nullptr;
  const long long before = g_launches.load();
  // capture on a private stream: the caller's may be the legacy default stream, which cannot
  // capture; the instantiated graph is then launched into the caller's stream
  static thread_local cudaStream_t cap_stream[64] = {};
  if (!cap_stream[dev.device])
    MMRS_CUDA(cudaStreamCreateWithFlags(&cap_stream[dev.device], cudaStreamNonBlocking));
  cudaStream_t cs = cap_stream[dev.device];
  MMRS_CUDA(cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal));
  const int rc = enqueue_search(a, dev, w, cs);
  const long long kernels = g_launches.load() - before;
  const cudaError_t ce = cudaStreamEndCapture(cs, &graph);
  if (rc != MMRS_OK) { if (graph) cudaGraphDestroy(graph); return rc; }
  if (ce != cudaSuccess) return fail(MMRS_ERR_CUDA, "cudaStreamEndCapture failed: %s", cudaGetErrorString(ce));
  const cudaError_t ie = cudaGraphInstantiate(&exec, graph, 0);
  if (ie != cudaSuccess) {
    cudaGraphDestroy(graph);
    return fail(MMRS_ERR_CUDA, "cudaGraphInstantiate failed: %s", cudaGetErrorString(ie));
  }
  GraphEntry e{key, graph, exec, ++g_graph_clock, kernels, {}, false, a.d_queries, a.d_values, a.d_indices, a.d_keys};
  e.patchable = discover_sites(graph, a, &e.sites);   // the graph is kept: its nodes own the parameter storage
  if (!e.patchable) { e.sites.clear(); g_stat_unpatchable.fetch_add(1); }
  g_stat_captures.fetch_add(1);
  if (g_graphs.size() >= kMaxGraphs) {   // evict the least recently used
    size_t victim = 0;
    for (size_t i = 1; i < g_graphs.size(); ++i)
      if (g_graphs[i].stamp < g_graphs[victim].stamp) victim = i;
    cudaGraphExecDestroy(g_graphs[victim].exec);
    cudaGraphDestroy(g_graphs[victim].graph);
    g_graphs.erase(g_graphs.begin() + victim);
  }
  g_graphs.push_back(e);
  MMRS_CUDA(cudaGraphLaunch(exec, stream));
  return MMRS_OK;
}

static int flags_to_status(int32_t f) {
  if (f & kFlagZeroNorm)
    return fail(MMRS_ERR_ZERO_NORM, "a query row has zero L2 norm and normalize_queries is set");
  if (f & kFlagGatherTimeout)
    return fail(MMRS_ERR_TIMEOUT, "fused all-gather: a peer rank did not deliver / acknowledge its top-k lists within "
                "MMRS_GATHER_TIMEOUT_MS (a dead or diverged rank; results of this batch are invalid)");
  if (f & kFlagWatchdog) return fail(MMRS_ERR_INTERNAL, "K2 pipeline watchdog fired (mbarrier wait timed out)");
  if (f & kFlagShort) return fail(MMRS_ERR_INTERNAL, "select saw fewer than k unique candidates");
  if (f & kFlagOverflow) return fail(MMRS_ERR_INTERNAL, "candidate list overflow");
  return MMRS_OK;
}

static int check_row_filter(const uint32_t* f) {
  if (reinterpret_cast<uintptr_t>(f) % sizeof(uint32_t) != 0)
    return fail(MMRS_ERR_ARG, "row filter pointer must be 4-byte aligned");
  return MMRS_OK;
}

// d_row_labels == NULL: unlabeled (the other two are ignored)
static int check_labels(const int32_t* row_labels, const int32_t* query_labels, int32_t label_match) {
  if (!row_labels) return MMRS_OK;
  if (!query_labels) return fail(MMRS_ERR_ARG, "row labels given without query labels");
  if (reinterpret_cast<uintptr_t>(row_labels) % sizeof(int32_t) != 0 ||
      reinterpret_cast<uintptr_t>(query_labels) % sizeof(int32_t) != 0)
    return fail(MMRS_ERR_ARG, "label pointers must be 4-byte aligned");
  if (label_match != MMRS_LABEL_SAME && label_match != MMRS_LABEL_OTHER)
    return fail(MMRS_ERR_ARG, "label_match %d must be MMRS_LABEL_SAME or MMRS_LABEL_OTHER", label_match);
  return MMRS_OK;
}

static int validate_search(const SearchArgs& a, const void* ws, size_t ws_bytes, size_t extra) {
  int rc = check_matrix(a.gallery, a.n_rows, a.dim, a.ld, a.dtype, "gallery");
  if (rc != MMRS_OK) return rc;
  if (a.n_queries < 0) return fail(MMRS_ERR_ARG, "n_queries < 0");
  if (a.k < 1 || a.k > 1024) return fail(MMRS_ERR_ARG, "k = %d must be in [1, 1024]", a.k);
  if (a.k > a.n_rows)
    return fail(MMRS_ERR_ARG, "k = %d exceeds the %lld gallery rows (torch.topk raises here too)",
                a.k, (long long)a.n_rows);
  if (a.ldq_in < a.dim) return fail(MMRS_ERR_ARG, "query row stride < dim");
  const size_t need = mmrs_search_workspace_bytes(a.n_rows, a.dim, a.dtype, a.n_queries, a.k) + extra;
  if (!ws || ws_bytes < need)
    return fail(MMRS_ERR_WORKSPACE, "workspace %zu bytes, need %zu", ws_bytes, need);
  if (reinterpret_cast<uintptr_t>(ws) % 256 != 0)
    return fail(MMRS_ERR_WORKSPACE, "workspace must be 256-byte aligned");
  return MMRS_OK;
}

}  // namespace mmrs

using namespace mmrs;

// the key merge of mmrs_topk_merge_keys_async / _padded_async (defined below)
static int merge_keys(const uint64_t* d_keys_in, int32_t n_lists, int32_t n_queries, int32_t k_in,
                      int64_t list_stride, int32_t k_out, float* d_out_values, int64_t* d_out_indices,
                      int32_t* d_status, int32_t* h_status, bool pad_short, void* stream_);

extern "C" {

int mmrs_abi_version(void) { return MMRS_ABI_VERSION; }
const char* mmrs_last_error(void) { return g_err; }

int mmrs_device_check(int device) {
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess)
    return fail(MMRS_ERR_CUDA, "cudaGetDeviceCount failed: %s", cudaGetErrorString(e));
  if (device < 0 || device >= count)
    return fail(MMRS_ERR_ARG, "device %d not present (%d visible)", device, count);
  int major = 0;
  MMRS_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
  if (major != 10)
    return fail(MMRS_ERR_ARCH, "device %d is compute capability %d.x; sm_100a required", device, major);
  return MMRS_OK;
}

size_t mmrs_full_scores_workspace_bytes(int64_t n_rows, int32_t dim, int32_t gallery_dtype,
                                        int32_t n_queries) {
  (void)gallery_dtype;
  return carve(nullptr, n_rows, dim, n_queries, 1, false).total;
}

int mmrs_full_scores(const void* d_gallery, int64_t n_rows, int32_t dim, int64_t ld_gallery,
                     int32_t gallery_dtype, const float* d_queries, int32_t n_queries,
                     int64_t ld_queries, int32_t normalize_queries, float scale, int32_t path,
                     float* d_out_scores, int64_t ld_out, void* d_workspace,
                     size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceInfo dev;
  int rc = current_device(&dev);
  if (rc != MMRS_OK) return rc;
  rc = check_matrix(d_gallery, n_rows, dim, ld_gallery, gallery_dtype, "gallery");
  if (rc != MMRS_OK) return rc;
  if (n_queries == 0) return MMRS_OK;
  if (n_queries < 0 || !d_queries || !d_out_scores || ld_out < n_rows || ld_queries < dim)
    return fail(MMRS_ERR_ARG, "bad query / output arguments");
  const size_t need = mmrs_full_scores_workspace_bytes(n_rows, dim, gallery_dtype, n_queries);
  if (!d_workspace || workspace_bytes < need || reinterpret_cast<uintptr_t>(d_workspace) % 256)
    return fail(MMRS_ERR_WORKSPACE, "workspace %zu bytes, need %zu (256-byte aligned)", workspace_bytes, need);
  const Workspace w = carve(d_workspace, n_rows, dim, n_queries, 1, false);
  const int32_t ldq = padded_dim(dim), qp = padded_queries(n_queries);
  const Path p = choose_path(path, gallery_dtype, n_queries);
  if (p == Path::kMma && gallery_dtype == MMRS_DTYPE_F32)
    return fail(MMRS_ERR_ARG, "MMRS_PATH_MMA needs a bf16 (or bf16x3) gallery");
  MMRS_CUDA(cudaMemsetAsync(w.flags, 0, 8 * sizeof(int32_t), stream));
  MMRS_LAUNCH(launch_prep_queries(d_queries, n_queries, ld_queries, dim, normalize_queries,
                                gallery_dtype == MMRS_DTYPE_BF16 ? 1 : (gallery_dtype == MMRS_DTYPE_BF16X3 ? 2 : 0),
                                w.q_f32, w.q_bf16, qp, ldq, w.flags, GatherPrologue{}, stream));
  ScanParams base{};
  base.gallery = d_gallery; base.n_rows = n_rows; base.ld = ld_gallery; base.dim = dim;
  base.queries = w.q_f32; base.ldq = ldq; base.scale = scale;
  base.out_scores = d_out_scores; base.ld_out = ld_out;
  const int32_t n_tiles = static_cast<int32_t>((n_rows + kTileRows - 1) / kTileRows);
  base.sched = TileSchedule{n_tiles, 1, 0, n_tiles};
  rc = run_scan(p, dev, gallery_dtype, base, w, qp, 0, n_queries, kModeScores, stream);
  if (rc != MMRS_OK) return rc;
  int32_t* h = pinned_status();
  if (!h) return fail(MMRS_ERR_CUDA, "cudaHostAlloc for the status word failed");
  MMRS_CUDA(cudaMemcpyAsync(h, w.flags, sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
  MMRS_CUDA(cudaStreamSynchronize(stream));
  return flags_to_status(h[0]);
}

int mmrs_split_bf16x3(const float* d_src, int64_t n_rows, int32_t dim, int64_t ld_src, void* d_dst,
                      int64_t ld_dst, void* stream) {
  DeviceInfo dev;
  int rc = current_device(&dev);
  if (rc != MMRS_OK) return rc;
  if (!d_src || !d_dst || n_rows < 1 || dim < 1 || ld_src < dim || ld_dst < dim || ld_dst % 8 != 0)
    return fail(MMRS_ERR_ARG, "bad arguments (ld_dst must be a multiple of 8 and >= dim)");
  MMRS_LAUNCH(launch_split_bf16x3(d_src, n_rows, dim, ld_src, static_cast<__nv_bfloat16*>(d_dst), ld_dst,
                                  dev.sm_count, static_cast<cudaStream_t>(stream)));
  return MMRS_OK;
}

size_t mmrs_search_workspace_bytes(int64_t n_rows, int32_t dim, int32_t gallery_dtype,
                                   int32_t n_queries, int32_t k) {
  (void)gallery_dtype;
  if (n_rows < 1 || dim < 1 || n_queries < 0 || k < 1) return 0;
  return carve(nullptr, n_rows, dim, n_queries < 1 ? 1 : n_queries, k, true).total;
}

size_t mmrs_search_host_staging_bytes(int32_t dim, int32_t n_queries, int32_t k) {
  if (n_queries < 1) n_queries = 1;
  return align_up(static_cast<size_t>(n_queries) * dim * sizeof(float), 256) +
         align_up(static_cast<size_t>(n_queries) * k * sizeof(float), 256) +
         align_up(static_cast<size_t>(n_queries) * k * sizeof(int64_t), 256);
}

// Validate, stage host queries (host_io), enqueue the search (graph replay) and the read-back of
// the status word -- and of the results when host_io -- on `stream`.  Nothing is synchronised.
static int search_enqueue(SearchArgs& a, const float* h_queries, float* h_values, int64_t* h_indices,
                          void* d_workspace, size_t workspace_bytes, int32_t* h_status,
                          cudaStream_t stream, DeviceInfo* dev_out, Workspace* w_out) {
  DeviceInfo dev;
  int rc = current_device(&dev);
  if (rc != MMRS_OK) return rc;
  const bool host_io = h_queries != nullptr;
  const size_t staging = host_io ? mmrs_search_host_staging_bytes(a.dim, a.n_queries, a.k) : 0;
  rc = validate_search(a, d_workspace, workspace_bytes, staging);
  if (rc != MMRS_OK) return rc;
  if (!h_status) return fail(MMRS_ERR_ARG, "null status pointer");
  h_status[0] = 0;
  if (a.n_queries == 0) return MMRS_OK;
  if (!host_io && (!a.d_queries || (!a.d_keys && a.g_world == 0 && (!a.d_values || !a.d_indices))))
    return fail(MMRS_ERR_ARG, "null query / output pointer");
  const Workspace w = carve(d_workspace, a.n_rows, a.dim, a.n_queries, a.k, true);
  const size_t vbytes = static_cast<size_t>(a.n_queries) * a.k * sizeof(float);
  const size_t ibytes = static_cast<size_t>(a.n_queries) * a.k * sizeof(int64_t);
  if (host_io) {
    if (!h_values || !h_indices) return fail(MMRS_ERR_ARG, "null host output pointer");
    char* s = static_cast<char*>(d_workspace) + w.total;
    float* dq = reinterpret_cast<float*>(s);
    s += align_up(static_cast<size_t>(a.n_queries) * a.dim * sizeof(float), 256);
    a.d_values = reinterpret_cast<float*>(s);
    s += align_up(vbytes, 256);
    a.d_indices = reinterpret_cast<int64_t*>(s);
    MMRS_CUDA(cudaMemcpy2DAsync(dq, static_cast<size_t>(a.dim) * sizeof(float), h_queries,
                                static_cast<size_t>(a.ldq_in) * sizeof(float),
                                static_cast<size_t>(a.dim) * sizeof(float), a.n_queries,
                                cudaMemcpyHostToDevice, stream));
    a.d_queries = dq;
    a.ldq_in = a.dim;
  }
  rc = launch_search_graph(a, dev, w, d_workspace, stream);
  if (rc != MMRS_OK) return rc;
  MMRS_CUDA(cudaMemcpyAsync(h_status, w.flags, sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
  if (host_io) {
    MMRS_CUDA(cudaMemcpyAsync(h_values, a.d_values, vbytes, cudaMemcpyDeviceToHost, stream));
    MMRS_CUDA(cudaMemcpyAsync(h_indices, a.d_indices, ibytes, cudaMemcpyDeviceToHost, stream));
  }
  if (dev_out) *dev_out = dev;
  if (w_out) *w_out = w;
  return MMRS_OK;
}

static int search_common(SearchArgs a, const float* h_queries, float* h_values, int64_t* h_indices,
                         void* d_workspace, size_t workspace_bytes, cudaStream_t stream) {
  int32_t* h = pinned_status();
  if (!h) return fail(MMRS_ERR_CUDA, "cudaHostAlloc for the status word failed");
  int rc = search_enqueue(a, h_queries, h_values, h_indices, d_workspace, workspace_bytes, h, stream, nullptr, nullptr);
  if (rc != MMRS_OK || a.n_queries == 0) return rc;
  MMRS_CUDA(cudaStreamSynchronize(stream));
  return mmrs_search_status(h);   // MMRS_ERR_RETRY on a candidate-list overflow: mmrs_search_topk_exhaustive
}

size_t mmrs_search_exhaustive_workspace_bytes(int64_t n_rows, int32_t dim, int32_t n_queries) {
  if (n_rows < 1 || dim < 1 || n_queries < 1) return 0;
  return carve(nullptr, n_rows, dim, n_queries, 1, true, true).total;
}

int mmrs_search_topk_exhaustive(const void* d_gallery, int64_t n_rows, int32_t dim, int64_t ld_gallery,
                                int32_t gallery_dtype, const float* d_queries, int32_t n_queries,
                                int64_t ld_queries, int32_t k, int32_t normalize_queries, float scale,
                                int64_t index_offset, float* d_out_values, int64_t* d_out_indices,
                                void* d_workspace, size_t workspace_bytes, void* stream) {
  return mmrs_search_topk_exhaustive_filtered(d_gallery, n_rows, dim, ld_gallery, gallery_dtype, d_queries, n_queries,
                                              ld_queries, k, normalize_queries, scale, index_offset, d_out_values,
                                              d_out_indices, d_workspace, workspace_bytes, nullptr, stream);
}

int mmrs_search_topk_exhaustive_filtered(const void* d_gallery, int64_t n_rows, int32_t dim, int64_t ld_gallery,
                                         int32_t gallery_dtype, const float* d_queries, int32_t n_queries,
                                         int64_t ld_queries, int32_t k, int32_t normalize_queries, float scale,
                                         int64_t index_offset, float* d_out_values, int64_t* d_out_indices,
                                         void* d_workspace, size_t workspace_bytes, const uint32_t* d_row_filter,
                                         void* stream) {
  return mmrs_search_topk_exhaustive_labeled(d_gallery, n_rows, dim, ld_gallery, gallery_dtype, d_queries, n_queries,
                                             ld_queries, k, normalize_queries, scale, index_offset, d_out_values,
                                             d_out_indices, d_workspace, workspace_bytes, d_row_filter, nullptr,
                                             nullptr, 0, stream);
}

int mmrs_search_topk_exhaustive_labeled(const void* d_gallery, int64_t n_rows, int32_t dim, int64_t ld_gallery,
                                        int32_t gallery_dtype, const float* d_queries, int32_t n_queries,
                                        int64_t ld_queries, int32_t k, int32_t normalize_queries, float scale,
                                        int64_t index_offset, float* d_out_values, int64_t* d_out_indices,
                                        void* d_workspace, size_t workspace_bytes, const uint32_t* d_row_filter,
                                        const int32_t* d_row_labels, const int32_t* d_query_labels,
                                        int32_t label_match, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceInfo dev;
  int rc = current_device(&dev);
  if (rc != MMRS_OK) return rc;
  rc = check_matrix(d_gallery, n_rows, dim, ld_gallery, gallery_dtype, "gallery");
  if (rc != MMRS_OK) return rc;
  if (n_queries == 0) return MMRS_OK;
  if (n_queries < 0 || !d_queries || !d_out_values || !d_out_indices || ld_queries < dim)
    return fail(MMRS_ERR_ARG, "bad query / output arguments");
  if (k < 1 || k > 1024 || k > n_rows) return fail(MMRS_ERR_ARG, "k = %d must be in [1, min(1024, n_rows)]", k);
  const size_t need = mmrs_search_exhaustive_workspace_bytes(n_rows, dim, n_queries);
  if (!d_workspace || workspace_bytes < need || reinterpret_cast<uintptr_t>(d_workspace) % 256)
    return fail(MMRS_ERR_WORKSPACE, "workspace %zu bytes, need %zu (256-byte aligned)", workspace_bytes, need);
  const Workspace w = carve(d_workspace, n_rows, dim, n_queries, 1, true, true);
  SearchArgs a{d_gallery, n_rows, dim, ld_gallery, gallery_dtype, d_queries, n_queries, ld_queries,
               k, normalize_queries, scale, index_offset, MMRS_PATH_AUTO, d_out_values, d_out_indices};
  a.row_filter = d_row_filter;
  a.row_labels = d_row_labels; a.query_labels = d_query_labels; a.label_match = label_match;
  rc = check_row_filter(d_row_filter);
  if (rc != MMRS_OK) return rc;
  rc = check_labels(d_row_labels, d_query_labels, label_match);
  if (rc != MMRS_OK) return rc;
  rc = enqueue_exhaustive(a, dev, w, stream);
  if (rc != MMRS_OK) return rc;
  int32_t* h = pinned_status();
  if (!h) return fail(MMRS_ERR_CUDA, "cudaHostAlloc for the status word failed");
  MMRS_CUDA(cudaMemcpyAsync(h, w.flags, sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
  MMRS_CUDA(cudaStreamSynchronize(stream));
  return flags_to_status(h[0]);
}

int mmrs_search_topk(const void* d_gallery, int64_t n_rows, int32_t dim, int64_t ld_gallery,
                     int32_t gallery_dtype, const float* d_queries, int32_t n_queries,
                     int64_t ld_queries, int32_t k, int32_t normalize_queries, float scale,
                     int64_t index_offset, int32_t path, float* d_out_values,
                     int64_t* d_out_indices, void* d_workspace, size_t workspace_bytes,
                     void* stream) {
  SearchArgs a{d_gallery, n_rows, dim, ld_gallery, gallery_dtype, d_queries, n_queries, ld_queries,
               k, normalize_queries, scale, index_offset, path, d_out_values, d_out_indices};
  return search_common(a, nullptr, nullptr, nullptr, d_workspace, workspace_bytes,
                       static_cast<cudaStream_t>(stream));
}

int mmrs_search_topk_host(const void* d_gallery, int64_t n_rows, int32_t dim, int64_t ld_gallery,
                          int32_t gallery_dtype, const float* h_queries, int32_t n_queries,
                          int64_t ld_queries, int32_t k, int32_t normalize_queries, float scale,
                          int64_t index_offset, int32_t path, float* h_out_values,
                          int64_t* h_out_indices, void* d_workspace, size_t workspace_bytes,
                          void* stream) {
  if (n_queries > 0 && !h_queries) return fail(MMRS_ERR_ARG, "null host query pointer");
  SearchArgs a{d_gallery, n_rows, dim, ld_gallery, gallery_dtype, nullptr, n_queries, ld_queries,
               k, normalize_queries, scale, index_offset, path, nullptr, nullptr};
  if (n_queries == 0) {
    static const float dummy = 0.f;
    h_queries = &dummy;
  }
  return search_common(a, h_queries, h_out_values, h_out_indices, d_workspace, workspace_bytes,
                       static_cast<cudaStream_t>(stream));
}

int mmrs_search_topk_async(const void* d_gallery, int64_t n_rows, int32_t dim, int64_t ld_gallery,
                           int32_t gallery_dtype, const float* d_queries, int32_t n_queries,
                           int64_t ld_queries, int32_t k, int32_t normalize_queries, float scale,
                           int64_t index_offset, int32_t path, float* d_out_values,
                           int64_t* d_out_indices, void* d_workspace, size_t workspace_bytes,
                           int32_t* h_status, void* stream) {
  return mmrs_search_topk_async_filtered(d_gallery, n_rows, dim, ld_gallery, gallery_dtype, d_queries, n_queries,
                                         ld_queries, k, normalize_queries, scale, index_offset, path, d_out_values,
                                         d_out_indices, d_workspace, workspace_bytes, h_status, nullptr, stream);
}

int mmrs_search_topk_async_filtered(const void* d_gallery, int64_t n_rows, int32_t dim, int64_t ld_gallery,
                                    int32_t gallery_dtype, const float* d_queries, int32_t n_queries,
                                    int64_t ld_queries, int32_t k, int32_t normalize_queries, float scale,
                                    int64_t index_offset, int32_t path, float* d_out_values,
                                    int64_t* d_out_indices, void* d_workspace, size_t workspace_bytes,
                                    int32_t* h_status, const uint32_t* d_row_filter, void* stream) {
  return mmrs_search_topk_async_labeled(d_gallery, n_rows, dim, ld_gallery, gallery_dtype, d_queries, n_queries,
                                        ld_queries, k, normalize_queries, scale, index_offset, path, d_out_values,
                                        d_out_indices, d_workspace, workspace_bytes, h_status, d_row_filter, nullptr,
                                        nullptr, 0, stream);
}

int mmrs_search_topk_async_labeled(const void* d_gallery, int64_t n_rows, int32_t dim, int64_t ld_gallery,
                                   int32_t gallery_dtype, const float* d_queries, int32_t n_queries,
                                   int64_t ld_queries, int32_t k, int32_t normalize_queries, float scale,
                                   int64_t index_offset, int32_t path, float* d_out_values,
                                   int64_t* d_out_indices, void* d_workspace, size_t workspace_bytes,
                                   int32_t* h_status, const uint32_t* d_row_filter, const int32_t* d_row_labels,
                                   const int32_t* d_query_labels, int32_t label_match, void* stream) {
  SearchArgs a{d_gallery, n_rows, dim, ld_gallery, gallery_dtype, d_queries, n_queries, ld_queries,
               k, normalize_queries, scale, index_offset, path, d_out_values, d_out_indices};
  a.row_filter = d_row_filter;
  a.row_labels = d_row_labels; a.query_labels = d_query_labels; a.label_match = label_match;
  int rc = check_row_filter(d_row_filter);
  if (rc != MMRS_OK) return rc;
  rc = check_labels(d_row_labels, d_query_labels, label_match);
  if (rc != MMRS_OK) return rc;
  return search_enqueue(a, nullptr, nullptr, nullptr, d_workspace, workspace_bytes, h_status,
                        static_cast<cudaStream_t>(stream), nullptr, nullptr);
}

int mmrs_search_topk_host_async(const void* d_gallery, int64_t n_rows, int32_t dim, int64_t ld_gallery,
                                int32_t gallery_dtype, const float* h_queries, int32_t n_queries,
                                int64_t ld_queries, int32_t k, int32_t normalize_queries, float scale,
                                int64_t index_offset, int32_t path, float* h_out_values,
                                int64_t* h_out_indices, void* d_workspace, size_t workspace_bytes,
                                int32_t* h_status, void* stream) {
  return mmrs_search_topk_host_async_filtered(d_gallery, n_rows, dim, ld_gallery, gallery_dtype, h_queries, n_queries,
                                              ld_queries, k, normalize_queries, scale, index_offset, path, h_out_values,
                                              h_out_indices, d_workspace, workspace_bytes, h_status, nullptr, stream);
}

int mmrs_search_topk_host_async_filtered(const void* d_gallery, int64_t n_rows, int32_t dim, int64_t ld_gallery,
                                         int32_t gallery_dtype, const float* h_queries, int32_t n_queries,
                                         int64_t ld_queries, int32_t k, int32_t normalize_queries, float scale,
                                         int64_t index_offset, int32_t path, float* h_out_values,
                                         int64_t* h_out_indices, void* d_workspace, size_t workspace_bytes,
                                         int32_t* h_status, const uint32_t* d_row_filter, void* stream) {
  return mmrs_search_topk_host_async_labeled(d_gallery, n_rows, dim, ld_gallery, gallery_dtype, h_queries, n_queries,
                                             ld_queries, k, normalize_queries, scale, index_offset, path, h_out_values,
                                             h_out_indices, d_workspace, workspace_bytes, h_status, d_row_filter,
                                             nullptr, nullptr, 0, stream);
}

int mmrs_search_topk_host_async_labeled(const void* d_gallery, int64_t n_rows, int32_t dim, int64_t ld_gallery,
                                        int32_t gallery_dtype, const float* h_queries, int32_t n_queries,
                                        int64_t ld_queries, int32_t k, int32_t normalize_queries, float scale,
                                        int64_t index_offset, int32_t path, float* h_out_values,
                                        int64_t* h_out_indices, void* d_workspace, size_t workspace_bytes,
                                        int32_t* h_status, const uint32_t* d_row_filter, const int32_t* d_row_labels,
                                        const int32_t* d_query_labels, int32_t label_match, void* stream) {
  if (n_queries > 0 && !h_queries) return fail(MMRS_ERR_ARG, "null host query pointer");
  int rc = check_row_filter(d_row_filter);
  if (rc != MMRS_OK) return rc;
  rc = check_labels(d_row_labels, d_query_labels, label_match);
  if (rc != MMRS_OK) return rc;
  SearchArgs a{d_gallery, n_rows, dim, ld_gallery, gallery_dtype, nullptr, n_queries, ld_queries,
               k, normalize_queries, scale, index_offset, path, nullptr, nullptr};
  a.row_filter = d_row_filter;
  a.row_labels = d_row_labels; a.query_labels = d_query_labels; a.label_match = label_match;
  static const float dummy = 0.f;
  if (n_queries == 0) h_queries = &dummy;
  return search_enqueue(a, h_queries, h_out_values, h_out_indices, d_workspace, workspace_bytes,
                        h_status, static_cast<cudaStream_t>(stream), nullptr, nullptr);
}

int mmrs_search_topk_keys_async(const void* d_gallery, int64_t n_rows, int32_t dim, int64_t ld_gallery,
                                int32_t gallery_dtype, const float* d_queries, int32_t n_queries,
                                int64_t ld_queries, int32_t k, int32_t normalize_queries, float scale,
                                int64_t index_offset, int32_t path, uint64_t* d_out_keys,
                                void* d_workspace, size_t workspace_bytes, int32_t* h_status,
                                void* stream) {
  return mmrs_search_topk_keys_async_filtered(d_gallery, n_rows, dim, ld_gallery, gallery_dtype, d_queries, n_queries,
                                              ld_queries, k, normalize_queries, scale, index_offset, path, d_out_keys,
                                              d_workspace, workspace_bytes, h_status, nullptr, stream);
}

int mmrs_search_topk_keys_async_filtered(const void* d_gallery, int64_t n_rows, int32_t dim, int64_t ld_gallery,
                                         int32_t gallery_dtype, const float* d_queries, int32_t n_queries,
                                         int64_t ld_queries, int32_t k, int32_t normalize_queries, float scale,
                                         int64_t index_offset, int32_t path, uint64_t* d_out_keys,
                                         void* d_workspace, size_t workspace_bytes, int32_t* h_status,
                                         const uint32_t* d_row_filter, void* stream) {
  return mmrs_search_topk_keys_async_labeled(d_gallery, n_rows, dim, ld_gallery, gallery_dtype, d_queries, n_queries,
                                             ld_queries, k, normalize_queries, scale, index_offset, path, d_out_keys,
                                             d_workspace, workspace_bytes, h_status, d_row_filter, nullptr, nullptr, 0,
                                             stream);
}

int mmrs_search_topk_keys_async_labeled(const void* d_gallery, int64_t n_rows, int32_t dim, int64_t ld_gallery,
                                        int32_t gallery_dtype, const float* d_queries, int32_t n_queries,
                                        int64_t ld_queries, int32_t k, int32_t normalize_queries, float scale,
                                        int64_t index_offset, int32_t path, uint64_t* d_out_keys,
                                        void* d_workspace, size_t workspace_bytes, int32_t* h_status,
                                        const uint32_t* d_row_filter, const int32_t* d_row_labels,
                                        const int32_t* d_query_labels, int32_t label_match, void* stream) {
  {
    int rc = check_row_filter(d_row_filter);
    if (rc != MMRS_OK) return rc;
    rc = check_labels(d_row_labels, d_query_labels, label_match);
    if (rc != MMRS_OK) return rc;
  }
  if (index_offset < 0 || index_offset + n_rows > 0x100000000ll)
    return fail(MMRS_ERR_ARG, "global row ids must fit 32 bits");
  SearchArgs a{d_gallery, n_rows, dim, ld_gallery, gallery_dtype, d_queries, n_queries, ld_queries,
               k, normalize_queries, scale, index_offset, path, nullptr, nullptr};
  a.d_keys = d_out_keys;
  a.row_filter = d_row_filter;
  a.row_labels = d_row_labels; a.query_labels = d_query_labels; a.label_match = label_match;
  if (!d_out_keys) return fail(MMRS_ERR_ARG, "null key output pointer");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  uint64_t* tail = d_out_keys + static_cast<int64_t>(n_queries < 0 ? 0 : n_queries) * k;
  MMRS_CUDA(cudaMemsetAsync(tail, 0, sizeof(uint64_t), st));
  Workspace w{};
  int rc = search_enqueue(a, nullptr, nullptr, nullptr, d_workspace, workspace_bytes, h_status, st, nullptr, &w);
  if (rc != MMRS_OK || n_queries == 0) return rc;
  // the shard's status word travels with its keys, so that after the all-gather every rank knows
  // whether ANY rank has to repeat the batch -- no second collective
  MMRS_CUDA(cudaMemcpyAsync(tail, w.flags, sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
  return MMRS_OK;
}

int mmrs_topk_merge_keys_async(const uint64_t* d_keys_in, int32_t n_lists, int32_t n_queries, int32_t k_in,
                               int64_t list_stride, int32_t k_out, float* d_out_values,
                               int64_t* d_out_indices, int32_t* d_status, int32_t* h_status,
                               void* stream) {
  return merge_keys(d_keys_in, n_lists, n_queries, k_in, list_stride, k_out, d_out_values, d_out_indices, d_status,
                    h_status, false, stream);
}

int mmrs_topk_merge_keys_padded_async(const uint64_t* d_keys_in, int32_t n_lists, int32_t n_queries, int32_t k_in,
                                      int64_t list_stride, int32_t k_out, float* d_out_values,
                                      int64_t* d_out_indices, int32_t* d_status, int32_t* h_status,
                                      void* stream) {
  return merge_keys(d_keys_in, n_lists, n_queries, k_in, list_stride, k_out, d_out_values, d_out_indices, d_status,
                    h_status, true, stream);
}

}  // extern "C"

static int merge_keys(const uint64_t* d_keys_in, int32_t n_lists, int32_t n_queries, int32_t k_in,
                      int64_t list_stride, int32_t k_out, float* d_out_values, int64_t* d_out_indices,
                      int32_t* d_status, int32_t* h_status, bool pad_short, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceInfo dev;
  int rc = current_device(&dev);
  if (rc != MMRS_OK) return rc;
  if (!h_status || !d_status) return fail(MMRS_ERR_ARG, "null status pointer");
  h_status[0] = 0;
  if (n_queries == 0) return MMRS_OK;
  if (n_lists < 1 || n_queries < 0 || k_in < 1 || k_out < 1 || k_out > 1024 ||
      static_cast<int64_t>(n_lists) * k_in < k_out)
    return fail(MMRS_ERR_ARG, "bad merge shape: %d lists x %d, k_out %d", n_lists, k_in, k_out);
  if (!d_keys_in || !d_out_values || !d_out_indices) return fail(MMRS_ERR_ARG, "null pointer");
  MMRS_CUDA(cudaMemsetAsync(d_status, 0, sizeof(int32_t), stream));
  SelectParams sp{};
  sp.cand = const_cast<uint64_t*>(d_keys_in);
  sp.cap = n_lists * k_in; sp.fixed_n = n_lists * k_in; sp.k = k_out; sp.final_pass = 1;
  sp.out_values = d_out_values; sp.out_indices = d_out_indices; sp.index_offset = 0; sp.flags = d_status;
  if (list_stride < static_cast<int64_t>(n_queries) * k_in) return fail(MMRS_ERR_ARG, "list_stride too small");
  sp.seg_len = k_in; sp.seg_stride = list_stride;
  sp.pad_short = pad_short;
  MMRS_LAUNCH(launch_select(sp, n_queries, stream));
  MMRS_CUDA(cudaMemcpyAsync(h_status, d_status, sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
  return MMRS_OK;
}

extern "C" {

int mmrs_search_topk_fused_gather_async(const void* d_gallery, int64_t n_rows, int32_t dim, int64_t ld_gallery,
                                        int32_t gallery_dtype, const float* d_queries, int32_t n_queries,
                                        int64_t ld_queries, int32_t k_local, int32_t k_out,
                                        int32_t normalize_queries, float scale, int64_t index_offset, int32_t path,
                                        uint64_t* const* d_peer_bufs, uint32_t* const* d_peer_flags,
                                        uint64_t* d_local_buf, uint32_t* d_local_flags, int32_t rank, int32_t world,
                                        int64_t list_stride, float* d_out_values, int64_t* d_out_indices,
                                        void* d_workspace, size_t workspace_bytes, int32_t* h_status, void* stream) {
  return mmrs_search_topk_fused_gather_async_filtered(
      d_gallery, n_rows, dim, ld_gallery, gallery_dtype, d_queries, n_queries, ld_queries, k_local, k_out,
      normalize_queries, scale, index_offset, path, d_peer_bufs, d_peer_flags, d_local_buf, d_local_flags, rank, world,
      list_stride, d_out_values, d_out_indices, d_workspace, workspace_bytes, h_status, nullptr, stream);
}

int mmrs_search_topk_fused_gather_async_filtered(
    const void* d_gallery, int64_t n_rows, int32_t dim, int64_t ld_gallery, int32_t gallery_dtype,
    const float* d_queries, int32_t n_queries, int64_t ld_queries, int32_t k_local, int32_t k_out,
    int32_t normalize_queries, float scale, int64_t index_offset, int32_t path, uint64_t* const* d_peer_bufs,
    uint32_t* const* d_peer_flags, uint64_t* d_local_buf, uint32_t* d_local_flags, int32_t rank, int32_t world,
    int64_t list_stride, float* d_out_values, int64_t* d_out_indices, void* d_workspace, size_t workspace_bytes,
    int32_t* h_status, const uint32_t* d_row_filter, void* stream) {
  return mmrs_search_topk_fused_gather_async_labeled(
      d_gallery, n_rows, dim, ld_gallery, gallery_dtype, d_queries, n_queries, ld_queries, k_local, k_out,
      normalize_queries, scale, index_offset, path, d_peer_bufs, d_peer_flags, d_local_buf, d_local_flags, rank, world,
      list_stride, d_out_values, d_out_indices, d_workspace, workspace_bytes, h_status, d_row_filter, nullptr, nullptr,
      0, stream);
}

int mmrs_search_topk_fused_gather_async_labeled(
    const void* d_gallery, int64_t n_rows, int32_t dim, int64_t ld_gallery, int32_t gallery_dtype,
    const float* d_queries, int32_t n_queries, int64_t ld_queries, int32_t k_local, int32_t k_out,
    int32_t normalize_queries, float scale, int64_t index_offset, int32_t path, uint64_t* const* d_peer_bufs,
    uint32_t* const* d_peer_flags, uint64_t* d_local_buf, uint32_t* d_local_flags, int32_t rank, int32_t world,
    int64_t list_stride, float* d_out_values, int64_t* d_out_indices, void* d_workspace, size_t workspace_bytes,
    int32_t* h_status, const uint32_t* d_row_filter, const int32_t* d_row_labels, const int32_t* d_query_labels,
    int32_t label_match, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  {
    int rc = check_row_filter(d_row_filter);
    if (rc != MMRS_OK) return rc;
    rc = check_labels(d_row_labels, d_query_labels, label_match);
    if (rc != MMRS_OK) return rc;
  }
  if (world < 1 || world > kMaxWorld || rank < 0 || rank >= world || !d_peer_bufs || !d_peer_flags || !d_local_buf ||
      !d_local_flags)
    return fail(MMRS_ERR_ARG, "bad rank / world / peer pointers");
  if (n_queries < 1 || n_queries > kSuperChunk)
    return fail(MMRS_ERR_ARG, "fused gather handles 1..%d queries per call", kSuperChunk);
  if (k_local < 1 || k_out < 1 || k_out > 1024 || static_cast<int64_t>(world) * k_local < k_out)
    return fail(MMRS_ERR_ARG, "bad k_local / k_out");
  if (list_stride < static_cast<int64_t>(n_queries) * k_local + 1)
    return fail(MMRS_ERR_ARG, "list_stride must be at least n_queries * k_local + 1");
  if (index_offset < 0 || index_offset + n_rows > 0x100000000ll)
    return fail(MMRS_ERR_ARG, "global row ids must fit 32 bits");
  if (!d_out_values || !d_out_indices || !h_status) return fail(MMRS_ERR_ARG, "null output pointer");
  SearchArgs a{d_gallery, n_rows, dim, ld_gallery, gallery_dtype, d_queries, n_queries, ld_queries,
               k_local, normalize_queries, scale, index_offset, path, d_out_values, d_out_indices};
  a.g_world = world; a.g_rank = rank; a.g_peer_bufs = d_peer_bufs; a.g_peer_flags = d_peer_flags;
  a.g_local_buf = d_local_buf; a.g_local_flags = d_local_flags;
  a.g_list_stride = list_stride; a.g_k_out = k_out; a.g_timeout_ns = gather_timeout_ns();
  a.row_filter = d_row_filter;
  a.row_labels = d_row_labels; a.query_labels = d_query_labels; a.label_match = label_match;
  for (int r = 0; r <= world + 1; ++r) h_status[r] = 0;
  Workspace w{};
  // ONE graph: prep (epoch bump + ack wait) -> scans / selects -> producer select -> wait -> merge select
  int rc = search_enqueue(a, nullptr, nullptr, nullptr, d_workspace, workspace_bytes, h_status + world + 1, stream,
                          nullptr, &w);
  if (rc != MMRS_OK) return rc;
  // every rank's status word (the merge select's private snapshot) and the merge's own flags
  MMRS_CUDA(cudaMemcpyAsync(h_status, w.gscratch + kGStatus, static_cast<size_t>(world + 1) * sizeof(int32_t),
                            cudaMemcpyDeviceToHost, stream));
  return MMRS_OK;
}

int mmrs_gather_status(const int32_t* h_status, int32_t world) {
  if (!h_status || world < 1) return fail(MMRS_ERR_ARG, "bad arguments");
  int32_t all = 0;
  for (int r = 0; r <= world; ++r) all |= h_status[r];
  if (all == kFlagOverflow)
    return fail(MMRS_ERR_RETRY, "a candidate list overflowed on some rank: every rank repeats the batch on the general path");
  return flags_to_status(all);
}

int mmrs_search_status(const int32_t* h_status) {
  if (!h_status) return fail(MMRS_ERR_ARG, "null status pointer");
  const int32_t f = h_status[0];
  if (f == kFlagOverflow)
    return fail(MMRS_ERR_RETRY, "a candidate list overflowed: repeat this batch through the synchronous entry point");
  return flags_to_status(f);
}

size_t mmrs_topk_merge_workspace_bytes(int32_t n_lists, int32_t n_queries, int32_t k_in) {
  if (n_lists < 1 || n_queries < 1 || k_in < 1) return 256;
  return align_up(8 * sizeof(int32_t), 256) +
         align_up(static_cast<size_t>(n_queries) * n_lists * k_in * sizeof(uint64_t), 256);
}

int mmrs_topk_merge(const float* d_values_in, const int64_t* d_indices_in, int32_t n_lists,
                    int32_t n_queries, int32_t k_in, int32_t k_out, float* d_out_values,
                    int64_t* d_out_indices, void* d_workspace, size_t workspace_bytes,
                    void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceInfo dev;
  int rc = current_device(&dev);
  if (rc != MMRS_OK) return rc;
  if (n_queries == 0) return MMRS_OK;
  if (n_lists < 1 || n_queries < 0 || k_in < 1 || k_out < 1 || k_out > 1024 ||
      static_cast<int64_t>(n_lists) * k_in < k_out)
    return fail(MMRS_ERR_ARG, "bad merge shape: %d lists x %d, k_out %d", n_lists, k_in, k_out);
  if (!d_values_in || !d_indices_in || !d_out_values || !d_out_indices)
    return fail(MMRS_ERR_ARG, "null pointer");
  const size_t need = mmrs_topk_merge_workspace_bytes(n_lists, n_queries, k_in);
  if (!d_workspace || workspace_bytes < need || reinterpret_cast<uintptr_t>(d_workspace) % 256)
    return fail(MMRS_ERR_WORKSPACE, "workspace %zu bytes, need %zu (256-byte aligned)", workspace_bytes, need);
  int32_t* flags = static_cast<int32_t*>(d_workspace);
  uint64_t* cand = reinterpret_cast<uint64_t*>(static_cast<char*>(d_workspace) + align_up(8 * sizeof(int32_t), 256));
  const int32_t cap = n_lists * k_in;
  MMRS_CUDA(cudaMemsetAsync(flags, 0, 8 * sizeof(int32_t), stream));
  MMRS_LAUNCH(launch_pack_keys(d_values_in, d_indices_in, n_lists, n_queries, k_in, cand, cap, stream));
  SelectParams sp{};
  sp.cand = cand; sp.cnt = nullptr; sp.thr = nullptr; sp.cap = cap; sp.fixed_n = cap;
  sp.k = k_out; sp.final_pass = 1; sp.out_values = d_out_values; sp.out_indices = d_out_indices;
  sp.index_offset = 0; sp.flags = flags;
  MMRS_LAUNCH(launch_select(sp, n_queries, stream));
  int32_t* h = pinned_status();
  if (!h) return fail(MMRS_ERR_CUDA, "cudaHostAlloc for the status word failed");
  MMRS_CUDA(cudaMemcpyAsync(h, flags, sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
  MMRS_CUDA(cudaStreamSynchronize(stream));
  return flags_to_status(h[0]);
}

size_t mmrs_selfjoin_workspace_bytes(int64_t n_rows, int32_t dim, int32_t dtype) {
  (void)n_rows; (void)dim; (void)dtype;
  return 0;   // the exact-mode join keeps everything in registers / shared memory: d_workspace may be NULL
}

int mmrs_selfjoin_pairs(const void* d_emb, int64_t n_rows, int32_t dim, int64_t ld_emb,
                        int32_t dtype, float threshold, int64_t row_begin, int64_t row_end,
                        int64_t* d_out_pairs, int64_t capacity, int64_t* d_out_count,
                        void* d_workspace, size_t workspace_bytes, void* stream_) {
  (void)d_workspace; (void)workspace_bytes;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceInfo dev;
  int rc = current_device(&dev);
  if (rc != MMRS_OK) return rc;
  rc = check_matrix(d_emb, n_rows, dim, ld_emb, dtype, "embeddings");
  if (rc != MMRS_OK) return rc;
  if (dtype != MMRS_DTYPE_F32) return fail(MMRS_ERR_ARG, "self-join exact mode takes fp32 embeddings");
  if (dim % 8 != 0) return fail(MMRS_ERR_ARG, "self-join dim must be a multiple of 8 (pad with zeros)");
  if (row_begin < 0 || row_end > n_rows || row_begin > row_end || row_begin % 128 != 0)
    return fail(MMRS_ERR_ARG, "row range [%lld, %lld) invalid (begin must be a multiple of 128)",
                (long long)row_begin, (long long)row_end);
  if (capacity < 0 || (capacity > 0 && !d_out_pairs) || !d_out_count)
    return fail(MMRS_ERR_ARG, "bad output arguments");
  MMRS_CUDA(cudaMemsetAsync(d_out_count, 0, sizeof(int64_t), stream));
  MMRS_LAUNCH(launch_selfjoin_f32(static_cast<const float*>(d_emb), n_rows, dim, ld_emb, threshold,
                                row_begin, row_end, d_out_pairs, capacity, d_out_count,
                                dev.sm_count, stream));
  int32_t* h = pinned_status();
  if (!h) return fail(MMRS_ERR_CUDA, "cudaHostAlloc for the status word failed");
  int64_t* h64 = reinterpret_cast<int64_t*>(h);
  MMRS_CUDA(cudaMemcpyAsync(h64, d_out_count, sizeof(int64_t), cudaMemcpyDeviceToHost, stream));
  MMRS_CUDA(cudaStreamSynchronize(stream));
  if (h64[0] > capacity)
    return fail(MMRS_ERR_CAPACITY, "%lld pairs found, capacity %lld", (long long)h64[0], (long long)capacity);
  return MMRS_OK;
}

int mmrs_pack_row_filter(const uint8_t* d_allowed, int64_t n_rows, uint32_t* d_words, int64_t n_words,
                         int64_t* d_count, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceInfo dev;
  int rc = current_device(&dev);
  if (rc != MMRS_OK) return rc;
  if (n_rows < 1 || !d_allowed || !d_words || !d_count) return fail(MMRS_ERR_ARG, "bad arguments");
  const int64_t need = (n_rows + kTileRows - 1) / kTileRows * (kTileRows / 32);
  if (n_words < need)
    return fail(MMRS_ERR_ARG, "%lld words, need %lld (whole %d-row tiles)", (long long)n_words, (long long)need, kTileRows);
  rc = check_row_filter(d_words);
  if (rc != MMRS_OK) return rc;
  MMRS_CUDA(cudaMemsetAsync(d_count, 0, sizeof(int64_t), stream));
  MMRS_LAUNCH(launch_pack_row_filter(d_allowed, n_rows, d_words, n_words, reinterpret_cast<unsigned long long*>(d_count),
                                     dev.sm_count, stream));
  return MMRS_OK;
}

int64_t mmrs_launch_count(void) { return g_launches.load(); }

int mmrs_graph_stats(int64_t* h_out4) {
  if (!h_out4) return fail(MMRS_ERR_ARG, "null pointer");
  h_out4[0] = g_stat_captures.load(); h_out4[1] = g_stat_replays.load();
  h_out4[2] = g_stat_patches.load(); h_out4[3] = g_stat_unpatchable.load();
  return MMRS_OK;
}

size_t mmrs_sort_pairs_workspace_bytes(int64_t n_pairs) {
  if (n_pairs < 1) n_pairs = 1;
  int64_t m = 1;
  while (m < n_pairs) m <<= 1;
  return static_cast<size_t>(m) * sizeof(uint64_t);
}

int mmrs_sort_pairs(int64_t* d_pairs, int64_t n_pairs, void* d_workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceInfo dev;
  int rc = current_device(&dev);
  if (rc != MMRS_OK) return rc;
  if (n_pairs < 0 || (n_pairs > 0 && !d_pairs)) return fail(MMRS_ERR_ARG, "bad arguments");
  if (n_pairs < 2) return MMRS_OK;
  if (!d_workspace || workspace_bytes < mmrs_sort_pairs_workspace_bytes(n_pairs))
    return fail(MMRS_ERR_WORKSPACE, "workspace too small");
  MMRS_LAUNCH(launch_sort_pairs(d_pairs, n_pairs, static_cast<uint64_t*>(d_workspace), stream));
  return MMRS_OK;
}

int mmrs_row_norm_range(const float* d_emb, int64_t n_rows, int32_t dim, int64_t ld, float* d_out_min_max, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceInfo dev;
  int rc = current_device(&dev);
  if (rc != MMRS_OK) return rc;
  if (!d_emb || !d_out_min_max || n_rows < 1 || dim < 1 || ld < dim) return fail(MMRS_ERR_ARG, "bad arguments");
  MMRS_LAUNCH(launch_row_norm_range(d_emb, n_rows, dim, ld, d_out_min_max, dev.sm_count, stream));
  return MMRS_OK;
}

int mmrs_profile_enable(int on) {
  g_prof_on.store(on ? 1 : 0);
  return MMRS_OK;
}

int mmrs_profile_read(float* h_ms, int32_t* h_kind, int64_t* h_bytes, int64_t* h_flops, int32_t cap) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  int n = 0;
  for (ProfRec& r : g_prof) {
    float ms = -1.f;
    if (cudaEventSynchronize(r.e1) == cudaSuccess) cudaEventElapsedTime(&ms, r.e0, r.e1);
    if (n < cap) {
      if (h_ms) h_ms[n] = ms;
      if (h_kind) h_kind[n] = r.kind;
      if (h_bytes) h_bytes[n] = r.bytes;
      if (h_flops) h_flops[n] = r.flops;
      ++n;
    }
    cudaEventDestroy(r.e0);
    cudaEventDestroy(r.e1);
  }
  g_prof.clear();
  return n;
}

size_t mmrs_selfjoin_tc_workspace_bytes(int64_t n_rows, int64_t cand_capacity) {
  if (n_rows < 1) n_rows = 1;
  if (cand_capacity < 1) cand_capacity = 1;
  return 512 + align_up(static_cast<size_t>(sjm_max_panels(n_rows) + 1) * sizeof(int64_t), 256) +
         align_up(static_cast<size_t>(cand_capacity) * 2 * sizeof(int64_t), 256);
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
  const size_t need = mmrs_selfjoin_tc_workspace_bytes(n_rows, cand_capacity);
  if (!d_workspace || workspace_bytes < need || reinterpret_cast<uintptr_t>(d_workspace) % 256)
    return fail(MMRS_ERR_WORKSPACE, "workspace %zu bytes, need %zu (256-byte aligned)", workspace_bytes, need);
  char* b = static_cast<char*>(d_workspace);
  int32_t* flags = reinterpret_cast<int32_t*>(b);
  unsigned long long* counts = reinterpret_cast<unsigned long long*>(b + 256);   // [0] pairs, [1] candidates
  int64_t* d_panel = reinterpret_cast<int64_t*>(b + 512);
  const int64_t max_panels = sjm_max_panels(n_rows);
  int64_t* cand = reinterpret_cast<int64_t*>(b + 512 + align_up(static_cast<size_t>(max_panels + 1) * sizeof(int64_t), 256));

  std::vector<int64_t> h_panel(static_cast<size_t>(max_panels) + 1);
  int32_t n_my = 0;
  const bool pair = sjm_pair_mode(n_rows, dim, world);
  const int64_t tiles = sjm_plan(n_rows, rank, world, pair, h_panel.data(), static_cast<int32_t>(max_panels), &n_my);
  MMRS_CUDA(cudaMemsetAsync(b, 0, 512, stream));
  MMRS_CUDA(cudaMemcpyAsync(d_panel, h_panel.data(), static_cast<size_t>(n_my + 1) * sizeof(int64_t),
                            cudaMemcpyHostToDevice, stream));
  MMRS_CUDA(cudaStreamSynchronize(stream));   // h_panel is pageable and goes out of scope
  MMRS_LAUNCH(launch_selfjoin_mma(static_cast<const __nv_bfloat16*>(d_emb_bf16), n_rows, dim, ld_bf16,
                                  threshold - margin, rank, world, pair, d_panel, n_my, tiles, cand, cand_capacity,
                                  counts + 1, flags, dev.sm_count, stream));
  int32_t* h = pinned_status();
  if (!h) return fail(MMRS_ERR_CUDA, "cudaHostAlloc for the status word failed");
  int64_t* h64 = reinterpret_cast<int64_t*>(h);      // 32 bytes: [0] pairs, [1] candidates, [2] flags
  MMRS_CUDA(cudaMemcpyAsync(h64 + 1, counts + 1, sizeof(int64_t), cudaMemcpyDeviceToHost, stream));
  MMRS_CUDA(cudaMemcpyAsync(h64 + 2, flags, sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
  MMRS_CUDA(cudaStreamSynchronize(stream));
  if (h[4] & kFlagWatchdog) return fail(MMRS_ERR_INTERNAL, "self-join pipeline watchdog fired");
  const int64_t n_cand = h64[1];
  h64[0] = 0;
  if (n_cand <= cand_capacity) {
    MMRS_LAUNCH(launch_selfjoin_recheck(cand, n_cand, d_emb_f32, ld_f32, dim, threshold, d_out_pairs, capacity,
                                        counts, stream));
    MMRS_CUDA(cudaMemcpyAsync(h64, counts, sizeof(int64_t), cudaMemcpyDeviceToHost, stream));
  }
  MMRS_CUDA(cudaMemcpyAsync(d_out_count, counts, 2 * sizeof(int64_t), cudaMemcpyDeviceToDevice, stream));
  MMRS_CUDA(cudaStreamSynchronize(stream));
  if (n_cand > cand_capacity)
    return fail(MMRS_ERR_CAPACITY, "%lld candidate pairs, candidate capacity %lld", (long long)n_cand,
                (long long)cand_capacity);
  if (h64[0] > capacity)
    return fail(MMRS_ERR_CAPACITY, "%lld pairs found, capacity %lld", (long long)h64[0], (long long)capacity);
  return MMRS_OK;
}

size_t mmrs_threshold_sweep_workspace_bytes(int32_t n_thresholds) {
  if (n_thresholds < 1) n_thresholds = 1;
  return align_up(sizeof(unsigned long long) * 2 * (static_cast<size_t>(n_thresholds) + 1), 256);
}

int mmrs_threshold_sweep(const float* d_pos, int64_t n_pos, const float* d_neg, int64_t n_neg,
                         const double* d_thresholds, int32_t n_thresholds, int64_t* d_out_counts,
                         void* d_workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceInfo dev;
  int rc = current_device(&dev);
  if (rc != MMRS_OK) return rc;
  if (n_thresholds < 1 || n_thresholds > 4096) return fail(MMRS_ERR_ARG, "n_thresholds must be in [1, 4096]");
  if (n_pos < 0 || n_neg < 0 || (n_pos > 0 && !d_pos) || (n_neg > 0 && !d_neg) || !d_thresholds || !d_out_counts)
    return fail(MMRS_ERR_ARG, "bad arguments");
  if (!d_workspace || workspace_bytes < mmrs_threshold_sweep_workspace_bytes(n_thresholds))
    return fail(MMRS_ERR_WORKSPACE, "workspace too small");
  MMRS_LAUNCH(launch_threshold_sweep(d_pos, n_pos, d_neg, n_neg, d_thresholds, n_thresholds,
                                   d_out_counts, static_cast<unsigned long long*>(d_workspace),
                                   dev.sm_count, stream));
  return MMRS_OK;
}

int mmrs_threshold_sweep_f64(const double* d_pos, int64_t n_pos, const double* d_neg, int64_t n_neg,
                             const double* d_thresholds, int32_t n_thresholds, int64_t* d_out_counts,
                             void* d_workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceInfo dev;
  int rc = current_device(&dev);
  if (rc != MMRS_OK) return rc;
  if (n_thresholds < 1 || n_thresholds > 4096) return fail(MMRS_ERR_ARG, "n_thresholds must be in [1, 4096]");
  if (n_pos < 0 || n_neg < 0 || (n_pos > 0 && !d_pos) || (n_neg > 0 && !d_neg) || !d_thresholds || !d_out_counts)
    return fail(MMRS_ERR_ARG, "bad arguments");
  if (!d_workspace || workspace_bytes < mmrs_threshold_sweep_workspace_bytes(n_thresholds))
    return fail(MMRS_ERR_WORKSPACE, "workspace too small");
  MMRS_LAUNCH(launch_threshold_sweep_f64(d_pos, n_pos, d_neg, n_neg, d_thresholds, n_thresholds,
                                       d_out_counts, static_cast<unsigned long long*>(d_workspace),
                                       dev.sm_count, stream));
  return MMRS_OK;
}

int mmrs_threshold_sweep_labeled(const float* d_scores, const int64_t* d_targets, int64_t label, int64_t n,
                                 int32_t n_thresholds, int32_t grid_f32, double* d_out_thresholds, int64_t* d_out_counts,
                                 void* d_workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceInfo dev;
  int rc = current_device(&dev);
  if (rc != MMRS_OK) return rc;
  if (n_thresholds < 1 || n_thresholds > 4096) return fail(MMRS_ERR_ARG, "n_thresholds must be in [1, 4096]");
  if (n < 1 || !d_scores || !d_targets || !d_out_thresholds || !d_out_counts) return fail(MMRS_ERR_ARG, "bad arguments");
  if (!d_workspace || workspace_bytes < mmrs_threshold_sweep_workspace_bytes(n_thresholds) + 256)
    return fail(MMRS_ERR_WORKSPACE, "workspace too small (need mmrs_threshold_sweep_workspace_bytes + 256)");
  char* b = static_cast<char*>(d_workspace);
  MMRS_LAUNCH(launch_threshold_sweep_labeled(d_scores, d_targets, label, n, n_thresholds, grid_f32, d_out_thresholds,
                                             d_out_counts, reinterpret_cast<unsigned long long*>(b + 256),
                                             reinterpret_cast<uint32_t*>(b), dev.sm_count, stream));
  return MMRS_OK;
}

size_t mmrs_threshold_sweep_batched_workspace_bytes(int32_t n_queries, int32_t n_thresholds) {
  if (n_queries < 1) n_queries = 1;
  if (n_thresholds < 1) n_thresholds = 1;
  return align_up(sizeof(unsigned long long) * 2 * (static_cast<size_t>(n_thresholds) + 1) * n_queries, 256);
}

int mmrs_score_range_batched(const float* d_scores, int64_t ld_scores, int32_t n_queries, int64_t n_rows,
                             const uint32_t* d_row_filter, uint32_t* d_range, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceInfo dev;
  int rc = current_device(&dev);
  if (rc != MMRS_OK) return rc;
  if (n_queries == 0 || n_rows == 0) return MMRS_OK;
  if (n_queries < 0 || n_rows < 0 || ld_scores < n_rows || !d_scores || !d_range) return fail(MMRS_ERR_ARG, "bad arguments");
  MMRS_LAUNCH(launch_score_range_batched(d_scores, ld_scores, n_queries, n_rows, d_row_filter, d_range, dev.sm_count,
                                         stream));
  return MMRS_OK;
}

int mmrs_threshold_sweep_batched(const float* d_scores, int64_t ld_scores, int32_t n_queries, int64_t n_rows,
                                 const int32_t* d_row_labels, const int32_t* d_query_labels,
                                 const uint32_t* d_row_filter, const uint32_t* d_range, int32_t n_thresholds,
                                 int32_t grid_f32, double* d_out_thresholds, int64_t* d_out_counts,
                                 int64_t* d_out_n_pos, void* d_workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceInfo dev;
  int rc = current_device(&dev);
  if (rc != MMRS_OK) return rc;
  if (n_thresholds < 1 || n_thresholds > 4096) return fail(MMRS_ERR_ARG, "n_thresholds must be in [1, 4096]");
  if (n_queries == 0) return MMRS_OK;
  if (n_queries < 0 || n_rows < 1 || ld_scores < n_rows || !d_scores || !d_row_labels || !d_query_labels || !d_range ||
      !d_out_thresholds || !d_out_counts || !d_out_n_pos)
    return fail(MMRS_ERR_ARG, "bad arguments");
  if (!d_workspace || workspace_bytes < mmrs_threshold_sweep_batched_workspace_bytes(n_queries, n_thresholds))
    return fail(MMRS_ERR_WORKSPACE, "workspace too small (need mmrs_threshold_sweep_batched_workspace_bytes)");
  MMRS_LAUNCH(launch_threshold_sweep_batched(d_scores, ld_scores, n_queries, n_rows, d_row_labels, d_query_labels,
                                             d_row_filter, d_range, n_thresholds, grid_f32, d_out_thresholds,
                                             d_out_counts, d_out_n_pos, static_cast<unsigned long long*>(d_workspace),
                                             dev.sm_count, stream));
  return MMRS_OK;
}

size_t mmrs_range_search_workspace_bytes(int64_t window_rows, int32_t dim, int32_t n_queries) {
  if (window_rows < kTileRows || window_rows % kTileRows != 0 || dim < 1 || n_queries < 1) return 0;
  return carve_range(nullptr, window_rows, dim, n_queries).total_bytes;
}

static int check_range_window(int64_t window_rows, int32_t n_queries, const void* d_workspace, size_t workspace_bytes,
                              int32_t dim) {
  if (window_rows < kTileRows || window_rows % kTileRows != 0 || window_rows > 0x7fffffffll)
    return fail(MMRS_ERR_ARG, "window_rows = %lld must be a positive multiple of %d below 2^31", (long long)window_rows,
                kTileRows);
  if (n_queries < 1 || n_queries > 65535) return fail(MMRS_ERR_ARG, "n_queries = %d must be in [1, 65535]", n_queries);
  const size_t need = mmrs_range_search_workspace_bytes(window_rows, dim, n_queries);
  if (!d_workspace || workspace_bytes < need || reinterpret_cast<uintptr_t>(d_workspace) % 256)
    return fail(MMRS_ERR_WORKSPACE, "workspace %zu bytes, need %zu (256-byte aligned)", workspace_bytes, need);
  return MMRS_OK;
}

int mmrs_range_search_window(const void* d_gallery, int64_t n_rows, int32_t dim, int64_t ld_gallery,
                             int32_t gallery_dtype, const float* d_queries, int32_t n_queries, int64_t ld_queries,
                             int32_t normalize_queries, float scale, int32_t path, const float* d_thresholds,
                             int64_t row_begin, int64_t window_rows, const uint32_t* d_row_filter,
                             const int32_t* d_row_labels, const int32_t* d_query_labels, int32_t label_match,
                             int64_t* h_counts, void* d_workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceInfo dev;
  int rc = current_device(&dev);
  if (rc != MMRS_OK) return rc;
  rc = check_matrix(d_gallery, n_rows, dim, ld_gallery, gallery_dtype, "gallery");
  if (rc != MMRS_OK) return rc;
  rc = check_range_window(window_rows, n_queries, d_workspace, workspace_bytes, dim);
  if (rc != MMRS_OK) return rc;
  if (row_begin < 0 || row_begin >= n_rows || row_begin % kTileRows != 0)
    return fail(MMRS_ERR_ARG, "row_begin = %lld must be a multiple of %d inside the %lld rows", (long long)row_begin,
                kTileRows, (long long)n_rows);
  if (!d_queries || ld_queries < dim || !d_thresholds || !h_counts) return fail(MMRS_ERR_ARG, "bad query / output arguments");
  rc = check_row_filter(d_row_filter);
  if (rc != MMRS_OK) return rc;
  rc = check_labels(d_row_labels, d_query_labels, label_match);
  if (rc != MMRS_OK) return rc;
  const Path p = choose_path(path, gallery_dtype, n_queries);
  if (p == Path::kMma && gallery_dtype == MMRS_DTYPE_F32)
    return fail(MMRS_ERR_ARG, "MMRS_PATH_MMA needs a bf16 (or bf16x3) gallery");
  const RangeWorkspace w = carve_range(d_workspace, window_rows, dim, n_queries);
  const int32_t ldq = padded_dim(dim), qp = padded_queries(n_queries);
  const int64_t rows = n_rows - row_begin < window_rows ? n_rows - row_begin : window_rows;
  const int64_t n_words = window_rows / 32;
  MMRS_CUDA(cudaMemsetAsync(w.base.flags, 0, 8 * sizeof(int32_t), stream));
  MMRS_CUDA(cudaMemsetAsync(w.cnt, 0, static_cast<size_t>(n_queries) * sizeof(uint32_t), stream));
  MMRS_LAUNCH(launch_fill_u32(w.cnt + n_queries, static_cast<uint32_t>(window_rows), kRangePadLists, stream));
  MMRS_CUDA(cudaMemsetAsync(w.bitmap, 0, static_cast<size_t>(n_queries) * n_words * sizeof(uint32_t), stream));
  MMRS_LAUNCH(launch_prep_queries(d_queries, n_queries, ld_queries, dim, normalize_queries,
                                gallery_dtype == MMRS_DTYPE_BF16 ? 1 : (gallery_dtype == MMRS_DTYPE_BF16X3 ? 2 : 0),
                                w.base.q_f32, w.base.q_bf16, qp, ldq, w.base.flags, GatherPrologue{}, stream));
  // the window is a view of the gallery, like a shard: rows [row_begin, row_begin + rows) as local rows 0..rows-1
  // (row_begin is a multiple of 128, so the view's bitmap words and labels start on whole tiles)
  const size_t elem = gallery_dtype == MMRS_DTYPE_F32 ? sizeof(float) : sizeof(__nv_bfloat16);
  ScanParams base{};
  base.gallery = static_cast<const char*>(d_gallery) + static_cast<size_t>(row_begin) * ld_gallery * elem;
  base.n_rows = rows; base.ld = ld_gallery; base.dim = dim;
  base.queries = w.base.q_f32; base.ldq = ldq; base.scale = scale;
  const int32_t n_tiles = static_cast<int32_t>((rows + kTileRows - 1) / kTileRows);
  base.sched = TileSchedule{n_tiles, 1, 0, n_tiles};
  // cap = window_rows >= rows: a list holds at most one key per row, so it cannot overflow
  base.cand = w.cand; base.cnt = w.cnt; base.thr = d_thresholds; base.cap = static_cast<int32_t>(window_rows);
  base.row_filter = d_row_filter ? d_row_filter + row_begin / 32 : nullptr;
  base.row_labels = d_row_labels ? d_row_labels + row_begin : nullptr;
  base.query_labels = d_row_labels ? d_query_labels : nullptr;
  base.label_match = d_row_labels ? label_match : 0;
  rc = run_scan(p, dev, gallery_dtype, base, w.base, qp, 0, n_queries, kModeFilter, stream, n_rows);
  if (rc != MMRS_OK) return rc;
  MMRS_LAUNCH(launch_range_mark_prefix(w.cand, window_rows, w.cnt, n_queries, w.bitmap, w.word_base, w.chunk_sum,
                                       w.total, dev.sm_count, stream));
  int32_t* h = pinned_status();
  if (!h) return fail(MMRS_ERR_CUDA, "cudaHostAlloc for the status word failed");
  MMRS_CUDA(cudaMemcpyAsync(h, w.base.flags, sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
  MMRS_CUDA(cudaMemcpyAsync(h_counts, w.total, static_cast<size_t>(n_queries) * sizeof(int64_t),
                            cudaMemcpyDeviceToHost, stream));
  MMRS_CUDA(cudaStreamSynchronize(stream));
  return flags_to_status(h[0]);
}

int mmrs_range_search_scatter(int32_t n_queries, int64_t window_rows, int32_t dim, const int64_t* d_out_offsets,
                              int64_t index_offset, float* d_out_values, int64_t* d_out_indices, void* d_workspace,
                              size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceInfo dev;
  int rc = current_device(&dev);
  if (rc != MMRS_OK) return rc;
  rc = check_range_window(window_rows, n_queries, d_workspace, workspace_bytes, dim);
  if (rc != MMRS_OK) return rc;
  if (!d_out_offsets || !d_out_values || !d_out_indices) return fail(MMRS_ERR_ARG, "null output pointer");
  const RangeWorkspace w = carve_range(d_workspace, window_rows, dim, n_queries);
  MMRS_LAUNCH(launch_range_scatter(w.cand, window_rows, w.cnt, n_queries, w.bitmap, w.word_base, d_out_offsets,
                                   index_offset, d_out_values, d_out_indices, dev.sm_count, stream));
  return MMRS_OK;
}


size_t mmrs_resolve_duplicates_workspace_bytes(int64_t n_items, int64_t n_order, int64_t n_pairs) {
  if (n_items < 0 || n_order < 0 || n_pairs < 0) return 0;
  return carve_resolve(nullptr, n_items, n_order, n_pairs).total_bytes;
}

int mmrs_resolve_duplicates(const int64_t* d_pairs, int64_t n_pairs, const int64_t* d_order, int64_t n_order,
                            int64_t n_items, int64_t* d_representative, int64_t* h_rounds, void* d_workspace,
                            size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceInfo dev;
  int rc = current_device(&dev);
  if (rc != MMRS_OK) return rc;
  if (n_items < 0 || n_items > 0x7fffffffll)
    return fail(MMRS_ERR_ARG, "n = %lld rows: the resolve takes 0 <= n < 2^31", (long long)n_items);
  if (n_order < 0 || n_order > 0x7fffffffll)
    return fail(MMRS_ERR_ARG, "order of %lld ids: at most 2^31 - 1", (long long)n_order);
  if (!d_order && n_order > n_items) return fail(MMRS_ERR_ARG, "a null order stands for the ids 0..n_order-1 <= n");
  if (n_pairs < 0 || (n_pairs > 0 && !d_pairs) || (n_items > 0 && !d_representative))
    return fail(MMRS_ERR_ARG, "bad pair / output arguments");
  const size_t need = mmrs_resolve_duplicates_workspace_bytes(n_items, n_order, n_pairs);
  if (!d_workspace || workspace_bytes < need || reinterpret_cast<uintptr_t>(d_workspace) % 256)
    return fail(MMRS_ERR_WORKSPACE, "workspace %zu bytes, need %zu (256-byte aligned)", workspace_bytes, need);
  int32_t* h = pinned_status();
  if (!h) return fail(MMRS_ERR_CUDA, "cudaHostAlloc for the status word failed");
  const ResolveWorkspace w = carve_resolve(d_workspace, n_items, n_order, n_pairs);
  uint32_t* cnt = reinterpret_cast<uint32_t*>(w.header + 1);
  uint32_t* range = reinterpret_cast<uint32_t*>(w.header + 4);
  MMRS_CUDA(cudaMemsetAsync(w.header, 0, 256, stream));
  MMRS_CUDA(cudaMemsetAsync(w.rank, 0xff, static_cast<size_t>(n_items) * sizeof(uint32_t), stream));
  MMRS_CUDA(cudaMemsetAsync(d_representative, 0xff, static_cast<size_t>(n_items) * sizeof(int64_t), stream));   // -1
  MMRS_CUDA(cudaMemsetAsync(w.res, 0xff, static_cast<size_t>(n_order) * sizeof(int32_t), stream));             // undecided
  MMRS_LAUNCH(launch_resolve_rank(d_order, n_order, n_items, w.rank, w.header, dev.sm_count, stream));
  MMRS_LAUNCH(launch_resolve_orient(d_pairs, n_pairs, n_items, w.rank, w.edges, w.header, dev.sm_count, stream));
  MMRS_LAUNCH(launch_sort_pairs(w.edges, n_pairs, w.sort, stream));
  MMRS_LAUNCH(launch_resolve_offsets(w.edges, n_pairs, n_order, w.off, w.cursor, dev.sm_count, stream));
  // round k reads worklist (k + 1) & 1 (round 0: every rank) and writes worklist k & 1
  int64_t known = n_order, rounds = 0, tail = 0;
  while (known > 0) {
    for (int b = 0; b < kResolveBatch; ++b, ++rounds) {
      const int o = static_cast<int>(rounds & 1), i = o ^ 1;
      MMRS_LAUNCH(launch_resolve_round(rounds ? w.wl[i] : nullptr, cnt + i, n_order, known, w.wl[o], cnt + o, w.off,
                                       w.edges, w.cursor, w.res, dev.sm_count, stream));
    }
    MMRS_CUDA(cudaMemcpyAsync(h, w.header, 8 * sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
    MMRS_CUDA(cudaStreamSynchronize(stream));
    if (h[0]) break;
    const int last = static_cast<int>((rounds - 1) & 1);
    const int64_t left = static_cast<uint32_t>(h[1 + last]);
    const int64_t decided = known - left;
    known = left;
    if (left > 0 && decided < kResolveBatch * kResolveTailBelow) {
      MMRS_LAUNCH(launch_resolve_tail(w.wl[last], cnt + last, left, range, w.off, w.edges, w.cursor, w.res,
                                      dev.sm_count, stream));
      tail = left;
      break;
    }
  }
  MMRS_LAUNCH(launch_resolve_map_back(d_order, n_order, n_items, w.res, d_representative, dev.sm_count, stream));
  MMRS_CUDA(cudaMemcpyAsync(h, w.header, sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
  MMRS_CUDA(cudaStreamSynchronize(stream));
  if (h_rounds) { h_rounds[0] = rounds; h_rounds[1] = tail; }
  if (h[0] & kResolvePairRange) return fail(MMRS_ERR_ARG, "a pair id is outside [0, %lld)", (long long)n_items);
  if (h[0] & kResolveOrderRange) return fail(MMRS_ERR_ARG, "an order id is outside [0, %lld)", (long long)n_items);
  if (h[0] & kResolveOrderRepeat) return fail(MMRS_ERR_ARG, "an id appears more than once in the order");
  return MMRS_OK;
}

}  // extern "C"
