// api.cu -- the search forms of the extern "C" boundary declared in include/mmrs_b200.h (top-k in all its
// forms, full scores, merges, range search, split / quantise / pack) and the library-wide entry points, with
// the host-side orchestration of a search: query preparation, the phase schedule of plan.h, kernel choice
// (K1 streaming GEMV for small batches, K2 tcgen05 for the rest), the status read-back and the exhaustive
// re-run of a query whose candidate list overflowed.  The self-join, threshold-sweep and duplicate-resolve
// entry points live beside their kernels (selfjoin.cu, selfjoin_mma.cu, dedup_resolve.cu).
#include <stdlib.h>

#include <tuple>

#include "host.h"
#include "plan.h"

namespace mmrs {

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

static int env_int(const char* name, int dflt) {
  const char* s = getenv(name);
  return (s && *s) ? atoi(s) : dflt;
}

bool pdl_enabled() {
  static const bool on = env_int("MMRS_NO_PDL", 0) == 0;
  return on;
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
  __nv_bfloat16* q_bf16;   // [Qp, ldq]; int8 gallery: the int8 query rows [Qp, ldq + 16] bytes (fit: ldq >= 16)
  float* thr;              // [Qs]
  uint32_t* cnt;           // [Qs]
  uint64_t* cand;          // [Qs, cap] (>= n_tiles * kTileRows keys for the exhaustive path)
  size_t cand_keys;
  uint32_t* gscratch;      // [kGScratch] fused all-gather bookkeeping, see below
};
// gscratch words: [0] epoch of the slot (bumped by the prep kernel of every fused call; the caller
// zero-fills a workspace once, before its first use) [1] producer CTA counter [2] consumer CTA counter
// [8, 8 + world) snapshot of the ranks' status words [8 + world] status of the merge select
constexpr int kGScratch = 128;
constexpr int kGStatus = 8;
constexpr int kMaxWorld = 64;

static Workspace carve(Carver& c, int64_t n_rows, int32_t dim, int32_t n_queries, int32_t k, bool with_lists,
                       bool exhaustive = false) {
  Workspace w{};
  const int32_t ldq = padded_dim(dim), qp = padded_queries(n_queries);
  w.flags = c.take<int32_t>(8 * sizeof(int32_t));
  w.gscratch = c.take<uint32_t>(kGScratch * sizeof(uint32_t));
  w.q_f32 = c.take<float>(static_cast<size_t>(qp) * ldq * sizeof(float));
  w.q_bf16 = c.take<__nv_bfloat16>(3 * static_cast<size_t>(qp) * ldq * sizeof(__nv_bfloat16));   // up to 3 planes
  if (with_lists) {
    const SearchPlan pl = plan_for(n_rows, k, n_queries);
    const int32_t qs = n_queries < kSuperChunk ? n_queries : kSuperChunk;
    w.thr = c.take<float>(static_cast<size_t>(qs) * sizeof(float));
    w.cnt = c.take<uint32_t>(static_cast<size_t>(qs) * sizeof(uint32_t));
    // the exhaustive re-run (one query at a time, every row a key) needs n_tiles * 128 keys -- 0.8 GB
    // at 100M rows -- and is carved only for mmrs_search_topk_exhaustive's own, temporary workspace
    size_t keys = exhaustive ? static_cast<size_t>(pl.n_tiles) * kTileRows : static_cast<size_t>(qs) * pl.cap;
    w.cand_keys = keys;
    w.cand = c.take<uint64_t>(keys * sizeof(uint64_t));
  }
  return w;
}

// mmrs_search_topk_host / _host_async: the device copies of the host queries and results, after the search's
// own workspace (mmrs_search_host_staging_bytes)
struct HostStaging {
  float* queries;    // [n_queries, dim]
  float* values;     // [n_queries, k]
  int64_t* indices;  // [n_queries, k]
};

static HostStaging carve_staging(Carver& c, int32_t dim, int32_t n_queries, int32_t k) {
  HostStaging s;
  s.queries = c.take<float>(static_cast<size_t>(n_queries) * dim * sizeof(float));
  s.values = c.take<float>(static_cast<size_t>(n_queries) * k * sizeof(float));
  s.indices = c.take<int64_t>(static_cast<size_t>(n_queries) * k * sizeof(int64_t));
  return s;
}

// mmrs_topk_merge: the flag word, then the packed keys of every list
struct MergeWorkspace {
  int32_t* flags;    // [8]
  uint64_t* cand;    // [n_queries, n_lists * k_in]
};

static MergeWorkspace carve_merge(Carver& c, int32_t n_lists, int32_t n_queries, int32_t k_in) {
  MergeWorkspace w;
  w.flags = c.take<int32_t>(8 * sizeof(int32_t));
  w.cand = c.take<uint64_t>(static_cast<size_t>(n_queries) * n_lists * k_in * sizeof(uint64_t));
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
};

static RangeWorkspace carve_range(Carver& c, int64_t window_rows, int32_t dim, int32_t n_queries) {
  RangeWorkspace r{};
  r.base = carve(c, window_rows, dim, n_queries, 1, false);
  const size_t q = static_cast<size_t>(n_queries), words = static_cast<size_t>(window_rows / 32);
  r.cnt = c.take<uint32_t>((q + kRangePadLists) * sizeof(uint32_t));
  r.cand = c.take<uint64_t>(q * static_cast<size_t>(window_rows) * sizeof(uint64_t));
  r.bitmap = c.take<uint32_t>(q * words * sizeof(uint32_t));
  r.word_base = c.take<uint32_t>(q * words * sizeof(uint32_t));
  r.chunk_sum = c.take<uint32_t>(q * static_cast<size_t>(range_chunks(window_rows / 32)) * sizeof(uint32_t));
  r.total = c.take<int64_t>(q * sizeof(int64_t));
  return r;
}

// mmrs_refine_topk: the prepared queries of carve(), then one key per (query, candidate)
struct RefineWorkspace {
  Workspace base;   // flags, q_f32, q_bf16
  uint64_t* keys;   // [n_queries, k_cand]
};

static RefineWorkspace carve_refine(Carver& c, int32_t dim, int32_t n_queries, int32_t k_cand) {
  RefineWorkspace r{};
  r.base = carve(c, 1, dim, n_queries, 1, false);
  r.keys = c.take<uint64_t>(static_cast<size_t>(n_queries) * k_cand * sizeof(uint64_t));
  return r;
}

enum class Path { kGemv, kMma };

static int choose_path(int32_t requested, int32_t dtype, int32_t n_queries, Path* path) {
  if (dtype == MMRS_DTYPE_BF16X3) *path = Path::kMma;   // split planes exist for the tensor cores only
  else if (requested == MMRS_PATH_GEMV) *path = Path::kGemv;
  else if (requested == MMRS_PATH_MMA) *path = Path::kMma;
  // measured on B200 (profiles/r01_tune3.log): K1 wins for 1-2 queries, K2 from 3 on
  else if ((dtype == MMRS_DTYPE_BF16 || dtype == MMRS_DTYPE_I8) && n_queries > 2) *path = Path::kMma;
  else *path = Path::kGemv;
  if (*path == Path::kMma && dtype == MMRS_DTYPE_F32)
    return fail(MMRS_ERR_ARG, "MMRS_PATH_MMA needs a bf16, bf16x3 or int8 gallery");
  return MMRS_OK;
}

template <typename F>
static int profiled_scan(int32_t kind, int32_t dtype, const ScanParams& p, cudaStream_t stream, F launch) {
  const int64_t rows = g_prof_on.load(std::memory_order_relaxed) ? rows_in_schedule(p.sched, p.n_rows) : 0;
  // int8: the codes and the 16-byte tail that holds the row's scale
  const int64_t row_bytes = dtype == MMRS_DTYPE_I8 ? p.dim + 16 : p.dim * (dtype == MMRS_DTYPE_BF16 ? 2 : (dtype == MMRS_DTYPE_BF16X3 ? 6 : 4));
  return profiled_launch(kind, rows * row_bytes, 2 * rows * p.dim * p.nq, stream, launch);
}

// The mode of the prep kernel for a gallery dtype: 1 bf16 rounding, 2 bf16x3 planes, 3 int8 rows, 0 fp32.
static int32_t prep_mode(int32_t dtype) {
  return dtype == MMRS_DTYPE_BF16 ? 1 : (dtype == MMRS_DTYPE_BF16X3 ? 2 : (dtype == MMRS_DTYPE_I8 ? 3 : 0));
}

// Enqueue the prep kernel: the caller's queries -> the prepared matrices of `w` that the scans read.
// gp: the fused all-gather's prologue (none by default).
static int enqueue_prep(const float* queries, int32_t n_queries, int64_t ld_queries, int32_t dim, int32_t normalize,
                        int32_t dtype, const Workspace& w, cudaStream_t stream,
                        const GatherPrologue& gp = GatherPrologue{}) {
  return profiled_launch(4, 0, 0, stream, [&]() {
    return launch_prep_queries(queries, n_queries, ld_queries, dim, normalize, prep_mode(dtype), w.q_f32, w.q_bf16,
                               padded_queries(n_queries), padded_dim(dim), w.flags, gp, stream);
  });
}

// The ScanParams every scan of a call starts from: the gallery, the prepared queries of `w`, the scale and a
// schedule over every tile.  The prepared queries are fp32 rows [Qp, ldq], or for an int8 gallery the int8
// query rows the prep kernel wrote into q_bf16 in the gallery's row format (ldq + 16 bytes apart, s_q at byte ldq).
static ScanParams scan_base(const void* gallery, int64_t n_rows, int32_t dim, int64_t ld, int32_t dtype,
                            const Workspace& w, float scale) {
  ScanParams p{};
  p.gallery = gallery; p.n_rows = n_rows; p.ld = ld; p.dim = dim;
  const int32_t ldq = padded_dim(dim);
  if (dtype == MMRS_DTYPE_I8) {
    p.queries = reinterpret_cast<const float*>(w.q_bf16);
    p.ldq = ldq + 16;
  } else {
    p.queries = w.q_f32;
    p.ldq = ldq;
  }
  p.scale = scale;
  const int32_t n_tiles = static_cast<int32_t>((n_rows + kTileRows - 1) / kTileRows);
  p.sched = TileSchedule{n_tiles, 1, 0, n_tiles};
  return p;
}

// The row filter and the labels a scan applies; without row labels the query labels and the match are ignored.
static void set_constraints(ScanParams& p, const uint32_t* row_filter, const int32_t* row_labels,
                            const int32_t* query_labels, int32_t label_match) {
  p.row_filter = row_filter;
  p.row_labels = row_labels;
  p.query_labels = row_labels ? query_labels : nullptr;
  p.label_match = row_labels ? label_match : 0;
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
        return launch_scan_mma(p, w.q_bf16, n_q_padded, mode, w.flags, dev.sm_count, stream, split, plane_rows,
                               dtype == MMRS_DTYPE_I8);
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
  const uint32_t* row_filter = nullptr;   // allow-list bitmap over the local rows (mmrs_pack_row_filter); nullptr = all
  // label-conditioned search (ScanParams): row labels over the local rows (nullptr = unlabeled), device
  // query labels [n_queries], MMRS_LABEL_SAME / MMRS_LABEL_OTHER
  const int32_t* row_labels = nullptr;
  const int32_t* query_labels = nullptr;
  int32_t label_match = 0;
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
  // a query may legitimately see fewer than k eligible rows: the selects pad instead of flagging
  bool pad_short() const { return row_filter != nullptr || row_labels != nullptr; }
};

static uint64_t gather_timeout_ns() {
  const int ms = env_int("MMRS_GATHER_TIMEOUT_MS", 20000);
  return static_cast<uint64_t>(ms < 1 ? 1 : ms) * 1000000ull;
}

// Enqueue the whole fused search on `stream`.  Results are valid iff the flag word stays 0.
static int enqueue_search(const SearchArgs& a, const DeviceInfo& dev, const Workspace& w,
                          cudaStream_t stream) {
  const SearchPlan pl = plan_for(a.n_rows, a.k, a.n_queries);
  const int32_t qp = padded_queries(a.n_queries);
  Path path;
  int rc = choose_path(a.path, a.dtype, a.n_queries, &path);
  if (rc != MMRS_OK) return rc;
  const bool fused = a.g_world > 0;

  MMRS_CUDA(cudaMemsetAsync(w.flags, 0, 8 * sizeof(int32_t), stream));
  if (fused)   // status snapshot + merge status of this call (the epoch and the CTA counters persist)
    MMRS_CUDA(cudaMemsetAsync(w.gscratch + kGStatus, 0, (kMaxWorld + 1) * sizeof(uint32_t), stream));
  GatherPrologue gp{};
  if (fused) {
    gp.epoch = w.gscratch; gp.ack_flags = a.g_local_flags + a.g_world; gp.world = a.g_world;
    gp.timeout_ns = a.g_timeout_ns;
  }
  rc = enqueue_prep(a.d_queries, a.n_queries, a.ldq_in, a.dim, a.normalize, a.dtype, w, stream, gp);
  if (rc != MMRS_OK) return rc;
  ScanParams base = scan_base(a.gallery, a.n_rows, a.dim, a.ld, a.dtype, w, a.scale);
  base.cap = pl.cap;
  set_constraints(base, a.row_filter, a.row_labels, a.query_labels, a.label_match);

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
      rc = run_scan(path, dev, a.dtype, base, w, qp, s0, s1, mode, stream);
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
    rc = profiled_launch(5, 0, 0, stream, [&]() {
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
  const int32_t all_rows = pl.n_tiles * kTileRows;
  ScanParams base = scan_base(a.gallery, a.n_rows, a.dim, a.ld, a.dtype, w, a.scale);
  base.cap = all_rows;
  // one query per pass below, with that query's own label (query_labels[q0])
  set_constraints(base, a.row_filter, a.row_labels, a.query_labels, a.label_match);
  MMRS_CUDA(cudaMemsetAsync(w.flags, 0, 8 * sizeof(int32_t), stream));
  {
    int rc = enqueue_prep(a.d_queries, a.n_queries, a.ldq_in, a.dim, a.normalize, a.dtype, w, stream);
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
  auto tie() const {
    return std::tie(gallery, n_rows, dim, ld, dtype, n_queries, ldq_in, k, normalize, scale, index_offset, path,
                    workspace, device, ratio_log2, dense_tiles, has_values, has_indices, has_keys, g_world, g_rank,
                    g_bufs, g_flags, g_local_buf, g_local_flags, g_stride, g_k_out, g_timeout_ns, knobs, row_filter,
                    row_labels, query_labels, label_match);
  }
  bool operator==(const GraphKey& o) const { return tie() == o.tie(); }
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
  if (f & kFlagBadCandidate) return fail(MMRS_ERR_ARG, "refine: a candidate row is outside [-1, n_rows)");
  if (f & kFlagZeroNorm)
    return fail(MMRS_ERR_ZERO_NORM, "a query row has zero L2 norm and normalize_queries is set");
  if (f & kFlagNonFinite)
    return fail(MMRS_ERR_NONFINITE, "a query row holds a NaN or an infinity: int8 quantisation refuses it");
  if (f & kFlagGatherTimeout)
    return fail(MMRS_ERR_TIMEOUT, "fused all-gather: a peer rank did not deliver / acknowledge its top-k lists within "
                "MMRS_GATHER_TIMEOUT_MS (a dead or diverged rank; results of this batch are invalid)");
  if (f & kFlagWatchdog) return fail(MMRS_ERR_INTERNAL, "K2 pipeline watchdog fired (mbarrier wait timed out)");
  if (f & kFlagShort) return fail(MMRS_ERR_INTERNAL, "select saw fewer than k unique candidates");
  if (f & kFlagOverflow) return fail(MMRS_ERR_INTERNAL, "candidate list overflow");
  return MMRS_OK;
}

// The end of a synchronous call: copy the device flag word back, wait for `stream`, map the flags to a status.
static int read_status(const int32_t* d_flags, cudaStream_t stream) {
  int32_t* h = pinned_status();
  if (!h) return fail(MMRS_ERR_CUDA, "cudaHostAlloc for the status word failed");
  MMRS_CUDA(cudaMemcpyAsync(h, d_flags, sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
  MMRS_CUDA(cudaStreamSynchronize(stream));
  return flags_to_status(h[0]);
}

static int check_row_filter(const uint32_t* f) {
  if (reinterpret_cast<uintptr_t>(f) % sizeof(uint32_t) != 0)
    return fail(MMRS_ERR_ARG, "row filter pointer must be 4-byte aligned");
  return MMRS_OK;
}

// The row filter and the labels of a call; d_row_labels == NULL: unlabeled (the other two are ignored)
static int check_constraints(const uint32_t* row_filter, const int32_t* row_labels, const int32_t* query_labels,
                             int32_t label_match) {
  int rc = check_row_filter(row_filter);
  if (rc != MMRS_OK || !row_labels) return rc;
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
  rc = check_workspace(ws, ws_bytes, mmrs_search_workspace_bytes(a.n_rows, a.dim, a.dtype, a.n_queries, a.k) + extra);
  if (rc != MMRS_OK) return rc;
  return check_constraints(a.row_filter, a.row_labels, a.query_labels, a.label_match);
}

}  // namespace mmrs

using namespace mmrs;

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
  Carver c(nullptr);
  carve(c, n_rows, dim, n_queries, 1, false);
  return c.off;
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
  rc = check_workspace(d_workspace, workspace_bytes,
                       mmrs_full_scores_workspace_bytes(n_rows, dim, gallery_dtype, n_queries));
  if (rc != MMRS_OK) return rc;
  Path p;
  rc = choose_path(path, gallery_dtype, n_queries, &p);
  if (rc != MMRS_OK) return rc;
  Carver c(d_workspace);
  const Workspace w = carve(c, n_rows, dim, n_queries, 1, false);
  MMRS_CUDA(cudaMemsetAsync(w.flags, 0, 8 * sizeof(int32_t), stream));
  rc = enqueue_prep(d_queries, n_queries, ld_queries, dim, normalize_queries, gallery_dtype, w, stream);
  if (rc != MMRS_OK) return rc;
  ScanParams base = scan_base(d_gallery, n_rows, dim, ld_gallery, gallery_dtype, w, scale);
  base.out_scores = d_out_scores; base.ld_out = ld_out;
  rc = run_scan(p, dev, gallery_dtype, base, w, padded_queries(n_queries), 0, n_queries, kModeScores, stream);
  if (rc != MMRS_OK) return rc;
  return read_status(w.flags, stream);
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

int mmrs_quantize_rows_i8(const void* d_src, int32_t src_dtype, int64_t n_rows, int32_t dim, int64_t ld_src,
                          void* d_dst, int64_t ld_dst, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceInfo dev;
  int rc = current_device(&dev);
  if (rc != MMRS_OK) return rc;
  if (src_dtype != MMRS_DTYPE_F32 && src_dtype != MMRS_DTYPE_BF16)
    return fail(MMRS_ERR_ARG, "quantise: source dtype %d must be MMRS_DTYPE_F32 or MMRS_DTYPE_BF16", src_dtype);
  const int64_t dp = (static_cast<int64_t>(dim) + 15) / 16 * 16;
  if (!d_src || !d_dst || n_rows < 0 || dim < 1 || ld_src < dim || ld_dst < dp + 16 || ld_dst % 16 != 0 ||
      reinterpret_cast<uintptr_t>(d_dst) % 16 != 0)
    return fail(MMRS_ERR_ARG, "quantise: bad arguments (ld_dst must be >= round_up(dim, 16) + 16, a multiple of 16, "
                "and d_dst 16-byte aligned)");
  if (n_rows == 0) return MMRS_OK;
  int32_t* h = pinned_status();
  if (!h) return fail(MMRS_ERR_CUDA, "cudaHostAlloc for the status word failed");
  // a transient device status word: the call owns no workspace and keeps no device memory
  int32_t* d_status = nullptr;
  MMRS_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&d_status), sizeof(int32_t), stream));
  MMRS_CUDA(cudaMemsetAsync(d_status, 0, sizeof(int32_t), stream));
  MMRS_LAUNCH(launch_quantize_rows_i8(d_src, src_dtype, n_rows, dim, ld_src, static_cast<int8_t*>(d_dst), ld_dst,
                                      d_status, dev.sm_count, stream));
  MMRS_CUDA(cudaMemcpyAsync(h, d_status, sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
  MMRS_CUDA(cudaFreeAsync(d_status, stream));
  MMRS_CUDA(cudaStreamSynchronize(stream));
  if (h[0]) return fail(MMRS_ERR_NONFINITE, "a row holds a NaN or an infinity: int8 quantisation refuses it");
  return MMRS_OK;
}

size_t mmrs_search_workspace_bytes(int64_t n_rows, int32_t dim, int32_t gallery_dtype,
                                   int32_t n_queries, int32_t k) {
  (void)gallery_dtype;
  if (n_rows < 1 || dim < 1 || n_queries < 0 || k < 1) return 0;
  Carver c(nullptr);
  carve(c, n_rows, dim, n_queries < 1 ? 1 : n_queries, k, true);
  return c.off;
}

size_t mmrs_search_host_staging_bytes(int32_t dim, int32_t n_queries, int32_t k) {
  if (n_queries < 1) n_queries = 1;
  Carver c(nullptr);
  carve_staging(c, dim, n_queries, k);
  return c.off;
}

// Validate, stage host queries (host_io), enqueue the search (graph replay) and the read-back of
// the status word -- and of the results when host_io -- on `stream`.  Nothing is synchronised.
static int search_enqueue(SearchArgs& a, const float* h_queries, float* h_values, int64_t* h_indices,
                          void* d_workspace, size_t workspace_bytes, int32_t* h_status,
                          cudaStream_t stream, Workspace* w_out) {
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
  Carver c(d_workspace);
  const Workspace w = carve(c, a.n_rows, a.dim, a.n_queries, a.k, true);
  const size_t vbytes = static_cast<size_t>(a.n_queries) * a.k * sizeof(float);
  const size_t ibytes = static_cast<size_t>(a.n_queries) * a.k * sizeof(int64_t);
  if (host_io) {
    if (!h_values || !h_indices) return fail(MMRS_ERR_ARG, "null host output pointer");
    const HostStaging s = carve_staging(c, a.dim, a.n_queries, a.k);
    MMRS_CUDA(cudaMemcpy2DAsync(s.queries, static_cast<size_t>(a.dim) * sizeof(float), h_queries,
                                static_cast<size_t>(a.ldq_in) * sizeof(float),
                                static_cast<size_t>(a.dim) * sizeof(float), a.n_queries,
                                cudaMemcpyHostToDevice, stream));
    a.d_queries = s.queries;
    a.ldq_in = a.dim;
    a.d_values = s.values;
    a.d_indices = s.indices;
  }
  rc = launch_search_graph(a, dev, w, d_workspace, stream);
  if (rc != MMRS_OK) return rc;
  MMRS_CUDA(cudaMemcpyAsync(h_status, w.flags, sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
  if (host_io) {
    MMRS_CUDA(cudaMemcpyAsync(h_values, a.d_values, vbytes, cudaMemcpyDeviceToHost, stream));
    MMRS_CUDA(cudaMemcpyAsync(h_indices, a.d_indices, ibytes, cudaMemcpyDeviceToHost, stream));
  }
  if (w_out) *w_out = w;
  return MMRS_OK;
}

static int search_common(SearchArgs a, const float* h_queries, float* h_values, int64_t* h_indices,
                         void* d_workspace, size_t workspace_bytes, cudaStream_t stream) {
  int32_t* h = pinned_status();
  if (!h) return fail(MMRS_ERR_CUDA, "cudaHostAlloc for the status word failed");
  int rc = search_enqueue(a, h_queries, h_values, h_indices, d_workspace, workspace_bytes, h, stream, nullptr);
  if (rc != MMRS_OK || a.n_queries == 0) return rc;
  MMRS_CUDA(cudaStreamSynchronize(stream));
  return mmrs_search_status(h);   // MMRS_ERR_RETRY on a candidate-list overflow: mmrs_search_topk_exhaustive
}

size_t mmrs_search_exhaustive_workspace_bytes(int64_t n_rows, int32_t dim, int32_t n_queries) {
  if (n_rows < 1 || dim < 1 || n_queries < 1) return 0;
  Carver c(nullptr);
  carve(c, n_rows, dim, n_queries, 1, true, true);
  return c.off;
}

int mmrs_search_topk_exhaustive(const void* d_gallery, int64_t n_rows, int32_t dim, int64_t ld_gallery,
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
  rc = check_workspace(d_workspace, workspace_bytes, mmrs_search_exhaustive_workspace_bytes(n_rows, dim, n_queries));
  if (rc != MMRS_OK) return rc;
  rc = check_constraints(d_row_filter, d_row_labels, d_query_labels, label_match);
  if (rc != MMRS_OK) return rc;
  Carver c(d_workspace);
  const Workspace w = carve(c, n_rows, dim, n_queries, 1, true, true);
  const SearchArgs a{d_gallery, n_rows, dim, ld_gallery, gallery_dtype, d_queries, n_queries, ld_queries,
                     k, normalize_queries, scale, index_offset, MMRS_PATH_AUTO, d_out_values, d_out_indices,
                     d_row_filter, d_row_labels, d_query_labels, label_match};
  rc = enqueue_exhaustive(a, dev, w, stream);
  if (rc != MMRS_OK) return rc;
  return read_status(w.flags, stream);
}

size_t mmrs_refine_workspace_bytes(int32_t dim, int32_t n_queries, int32_t k_cand) {
  if (dim < 1 || n_queries < 1 || k_cand < 1) return 0;
  Carver c(nullptr);
  carve_refine(c, dim, n_queries, k_cand);
  return c.off;
}

int mmrs_refine_topk(const void* d_store, int32_t store_dtype, int64_t n_rows, int32_t dim, int64_t ld_store,
                     const float* d_queries, int32_t n_queries, int64_t ld_queries, int32_t normalize_queries,
                     float scale, const int64_t* d_candidates, int32_t k_cand, int64_t index_offset, int32_t k,
                     float* d_out_values, int64_t* d_out_indices, void* d_workspace, size_t workspace_bytes,
                     int32_t* h_status, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceInfo dev;
  int rc = current_device(&dev);
  if (rc != MMRS_OK) return rc;
  if (store_dtype != MMRS_DTYPE_F32 && store_dtype != MMRS_DTYPE_BF16)
    return fail(MMRS_ERR_ARG, "refine: store dtype %d must be MMRS_DTYPE_F32 or MMRS_DTYPE_BF16", store_dtype);
  rc = check_matrix(d_store, n_rows, dim, ld_store, store_dtype, "refine store");
  if (rc != MMRS_OK) return rc;
  if (h_status) h_status[0] = 0;
  if (n_queries == 0) return MMRS_OK;
  if (n_queries < 0 || !d_queries || !d_candidates || !d_out_values || !d_out_indices || ld_queries < dim)
    return fail(MMRS_ERR_ARG, "bad query / candidate / output arguments");
  if (k_cand < 1 || k < 1 || k > 1024 || k > k_cand)
    return fail(MMRS_ERR_ARG, "refine: k = %d must be in [1, min(1024, k_cand = %d)]", k, k_cand);
  rc = check_workspace(d_workspace, workspace_bytes, mmrs_refine_workspace_bytes(dim, n_queries, k_cand));
  if (rc != MMRS_OK) return rc;
  Carver c(d_workspace);
  const RefineWorkspace w = carve_refine(c, dim, n_queries, k_cand);
  MMRS_CUDA(cudaMemsetAsync(w.base.flags, 0, 8 * sizeof(int32_t), stream));
  rc = enqueue_prep(d_queries, n_queries, ld_queries, dim, normalize_queries, store_dtype, w.base, stream);
  if (rc != MMRS_OK) return rc;
  MMRS_LAUNCH(launch_refine_scores(d_store, store_dtype, n_rows, ld_store, dim, w.base.q_f32, padded_dim(dim), scale,
                                   d_candidates, n_queries, k_cand, w.keys, w.base.flags, stream));
  // the k best keys of each list; a list with fewer than k candidates (-1 entries) is padded with -inf / -1
  SelectParams sp{};
  sp.cand = w.keys; sp.cap = k_cand; sp.fixed_n = k_cand; sp.k = k; sp.final_pass = 1;
  sp.out_values = d_out_values; sp.out_indices = d_out_indices; sp.index_offset = index_offset;
  sp.flags = w.base.flags; sp.pad_short = 1;
  MMRS_LAUNCH(launch_select(sp, n_queries, stream));
  if (h_status) {
    MMRS_CUDA(cudaMemcpyAsync(h_status, w.base.flags, sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
    return MMRS_OK;
  }
  return read_status(w.base.flags, stream);
}

int mmrs_host_register(void* h_ptr, size_t bytes, void** d_ptr_out) {
  if (!h_ptr || bytes == 0 || !d_ptr_out) return fail(MMRS_ERR_ARG, "host register: null pointer or zero bytes");
  // a refused registration (e.g. pages already registered) is not sticky: clear it, or the next launcher's
  // cudaGetLastError() would report it
  cudaError_t e = cudaHostRegister(h_ptr, bytes, cudaHostRegisterPortable | cudaHostRegisterMapped);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return fail(MMRS_ERR_CUDA, "cudaHostRegister of %zu bytes failed: %s", bytes, cudaGetErrorString(e));
  }
  e = cudaHostGetDevicePointer(d_ptr_out, h_ptr, 0);
  if (e != cudaSuccess) {
    cudaHostUnregister(h_ptr);
    cudaGetLastError();
    return fail(MMRS_ERR_CUDA, "cudaHostGetDevicePointer failed: %s", cudaGetErrorString(e));
  }
  return MMRS_OK;
}

int mmrs_host_unregister(void* h_ptr) {
  if (!h_ptr) return fail(MMRS_ERR_ARG, "host unregister: null pointer");
  const cudaError_t e = cudaHostUnregister(h_ptr);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return fail(MMRS_ERR_CUDA, "cudaHostUnregister failed: %s", cudaGetErrorString(e));
  }
  return MMRS_OK;
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
                           int32_t* h_status, const uint32_t* d_row_filter, const int32_t* d_row_labels,
                           const int32_t* d_query_labels, int32_t label_match, void* stream) {
  SearchArgs a{d_gallery, n_rows, dim, ld_gallery, gallery_dtype, d_queries, n_queries, ld_queries,
               k, normalize_queries, scale, index_offset, path, d_out_values, d_out_indices,
               d_row_filter, d_row_labels, d_query_labels, label_match};
  return search_enqueue(a, nullptr, nullptr, nullptr, d_workspace, workspace_bytes, h_status,
                        static_cast<cudaStream_t>(stream), nullptr);
}

int mmrs_search_topk_host_async(const void* d_gallery, int64_t n_rows, int32_t dim, int64_t ld_gallery,
                                int32_t gallery_dtype, const float* h_queries, int32_t n_queries,
                                int64_t ld_queries, int32_t k, int32_t normalize_queries, float scale,
                                int64_t index_offset, int32_t path, float* h_out_values,
                                int64_t* h_out_indices, void* d_workspace, size_t workspace_bytes,
                                int32_t* h_status, const uint32_t* d_row_filter, const int32_t* d_row_labels,
                                const int32_t* d_query_labels, int32_t label_match, void* stream) {
  if (n_queries > 0 && !h_queries) return fail(MMRS_ERR_ARG, "null host query pointer");
  SearchArgs a{d_gallery, n_rows, dim, ld_gallery, gallery_dtype, nullptr, n_queries, ld_queries,
               k, normalize_queries, scale, index_offset, path, nullptr, nullptr,
               d_row_filter, d_row_labels, d_query_labels, label_match};
  static const float dummy = 0.f;
  if (n_queries == 0) h_queries = &dummy;
  return search_enqueue(a, h_queries, h_out_values, h_out_indices, d_workspace, workspace_bytes,
                        h_status, static_cast<cudaStream_t>(stream), nullptr);
}

int mmrs_search_topk_keys_async(const void* d_gallery, int64_t n_rows, int32_t dim, int64_t ld_gallery,
                                int32_t gallery_dtype, const float* d_queries, int32_t n_queries,
                                int64_t ld_queries, int32_t k, int32_t normalize_queries, float scale,
                                int64_t index_offset, int32_t path, uint64_t* d_out_keys,
                                void* d_workspace, size_t workspace_bytes, int32_t* h_status,
                                const uint32_t* d_row_filter, const int32_t* d_row_labels,
                                const int32_t* d_query_labels, int32_t label_match, void* stream) {
  if (index_offset < 0 || index_offset + n_rows > 0x100000000ll)
    return fail(MMRS_ERR_ARG, "global row ids must fit 32 bits");
  SearchArgs a{d_gallery, n_rows, dim, ld_gallery, gallery_dtype, d_queries, n_queries, ld_queries,
               k, normalize_queries, scale, index_offset, path, nullptr, nullptr,
               d_row_filter, d_row_labels, d_query_labels, label_match};
  a.d_keys = d_out_keys;
  if (!d_out_keys) return fail(MMRS_ERR_ARG, "null key output pointer");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  uint64_t* tail = d_out_keys + static_cast<int64_t>(n_queries < 0 ? 0 : n_queries) * k;
  MMRS_CUDA(cudaMemsetAsync(tail, 0, sizeof(uint64_t), st));
  Workspace w{};
  int rc = search_enqueue(a, nullptr, nullptr, nullptr, d_workspace, workspace_bytes, h_status, st, &w);
  if (rc != MMRS_OK || n_queries == 0) return rc;
  // the shard's status word travels with its keys, so that after the all-gather every rank knows
  // whether ANY rank has to repeat the batch -- no second collective
  MMRS_CUDA(cudaMemcpyAsync(tail, w.flags, sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
  return MMRS_OK;
}

int mmrs_topk_merge_keys_async(const uint64_t* d_keys_in, int32_t n_lists, int32_t n_queries, int32_t k_in,
                               int64_t list_stride, int32_t k_out, float* d_out_values,
                               int64_t* d_out_indices, int32_t* d_status, int32_t* h_status,
                               int32_t pad_short, void* stream_) {
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
  sp.pad_short = pad_short != 0;
  MMRS_LAUNCH(launch_select(sp, n_queries, stream));
  MMRS_CUDA(cudaMemcpyAsync(h_status, d_status, sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
  return MMRS_OK;
}

int mmrs_search_topk_fused_gather_async(
    const void* d_gallery, int64_t n_rows, int32_t dim, int64_t ld_gallery, int32_t gallery_dtype,
    const float* d_queries, int32_t n_queries, int64_t ld_queries, int32_t k_local, int32_t k_out,
    int32_t normalize_queries, float scale, int64_t index_offset, int32_t path, uint64_t* const* d_peer_bufs,
    uint32_t* const* d_peer_flags, uint64_t* d_local_buf, uint32_t* d_local_flags, int32_t rank, int32_t world,
    int64_t list_stride, float* d_out_values, int64_t* d_out_indices, void* d_workspace, size_t workspace_bytes,
    int32_t* h_status, const uint32_t* d_row_filter, const int32_t* d_row_labels, const int32_t* d_query_labels,
    int32_t label_match, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
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
               k_local, normalize_queries, scale, index_offset, path, d_out_values, d_out_indices,
               d_row_filter, d_row_labels, d_query_labels, label_match};
  a.g_world = world; a.g_rank = rank; a.g_peer_bufs = d_peer_bufs; a.g_peer_flags = d_peer_flags;
  a.g_local_buf = d_local_buf; a.g_local_flags = d_local_flags;
  a.g_list_stride = list_stride; a.g_k_out = k_out; a.g_timeout_ns = gather_timeout_ns();
  for (int r = 0; r <= world + 1; ++r) h_status[r] = 0;
  Workspace w{};
  // ONE graph: prep (epoch bump + ack wait) -> scans / selects -> producer select -> wait -> merge select
  int rc = search_enqueue(a, nullptr, nullptr, nullptr, d_workspace, workspace_bytes, h_status + world + 1, stream, &w);
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
  Carver c(nullptr);
  carve_merge(c, n_lists, n_queries, k_in);
  return c.off;
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
  rc = check_workspace(d_workspace, workspace_bytes, mmrs_topk_merge_workspace_bytes(n_lists, n_queries, k_in));
  if (rc != MMRS_OK) return rc;
  Carver c(d_workspace);
  const MergeWorkspace w = carve_merge(c, n_lists, n_queries, k_in);
  const int32_t cap = n_lists * k_in;
  MMRS_CUDA(cudaMemsetAsync(w.flags, 0, 8 * sizeof(int32_t), stream));
  MMRS_LAUNCH(launch_pack_keys(d_values_in, d_indices_in, n_lists, n_queries, k_in, w.cand, cap, stream));
  SelectParams sp{};
  sp.cand = w.cand; sp.cnt = nullptr; sp.thr = nullptr; sp.cap = cap; sp.fixed_n = cap;
  sp.k = k_out; sp.final_pass = 1; sp.out_values = d_out_values; sp.out_indices = d_out_indices;
  sp.index_offset = 0; sp.flags = w.flags;
  MMRS_LAUNCH(launch_select(sp, n_queries, stream));
  return read_status(w.flags, stream);
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

size_t mmrs_range_search_workspace_bytes(int64_t window_rows, int32_t dim, int32_t n_queries) {
  if (window_rows < kTileRows || window_rows % kTileRows != 0 || dim < 1 || n_queries < 1) return 0;
  Carver c(nullptr);
  carve_range(c, window_rows, dim, n_queries);
  return c.off;
}

static int check_range_window(int64_t window_rows, int32_t n_queries, const void* d_workspace, size_t workspace_bytes,
                              int32_t dim) {
  if (window_rows < kTileRows || window_rows % kTileRows != 0 || window_rows > 0x7fffffffll)
    return fail(MMRS_ERR_ARG, "window_rows = %lld must be a positive multiple of %d below 2^31", (long long)window_rows,
                kTileRows);
  if (n_queries < 1 || n_queries > 65535) return fail(MMRS_ERR_ARG, "n_queries = %d must be in [1, 65535]", n_queries);
  return check_workspace(d_workspace, workspace_bytes, mmrs_range_search_workspace_bytes(window_rows, dim, n_queries));
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
  rc = check_constraints(d_row_filter, d_row_labels, d_query_labels, label_match);
  if (rc != MMRS_OK) return rc;
  Path p;
  rc = choose_path(path, gallery_dtype, n_queries, &p);
  if (rc != MMRS_OK) return rc;
  Carver c(d_workspace);
  const RangeWorkspace w = carve_range(c, window_rows, dim, n_queries);
  const int64_t rows = n_rows - row_begin < window_rows ? n_rows - row_begin : window_rows;
  const int64_t n_words = window_rows / 32;
  MMRS_CUDA(cudaMemsetAsync(w.base.flags, 0, 8 * sizeof(int32_t), stream));
  MMRS_CUDA(cudaMemsetAsync(w.cnt, 0, static_cast<size_t>(n_queries) * sizeof(uint32_t), stream));
  MMRS_LAUNCH(launch_fill_u32(w.cnt + n_queries, static_cast<uint32_t>(window_rows), kRangePadLists, stream));
  MMRS_CUDA(cudaMemsetAsync(w.bitmap, 0, static_cast<size_t>(n_queries) * n_words * sizeof(uint32_t), stream));
  rc = enqueue_prep(d_queries, n_queries, ld_queries, dim, normalize_queries, gallery_dtype, w.base, stream);
  if (rc != MMRS_OK) return rc;
  // the window is a view of the gallery, like a shard: rows [row_begin, row_begin + rows) as local rows 0..rows-1
  // (row_begin is a multiple of 128, so the view's bitmap words and labels start on whole tiles)
  const size_t elem = gallery_dtype == MMRS_DTYPE_F32 ? sizeof(float) : (gallery_dtype == MMRS_DTYPE_I8 ? 1 : sizeof(__nv_bfloat16));
  ScanParams base = scan_base(static_cast<const char*>(d_gallery) + static_cast<size_t>(row_begin) * ld_gallery * elem,
                              rows, dim, ld_gallery, gallery_dtype, w.base, scale);
  // cap = window_rows >= rows: a list holds at most one key per row, so it cannot overflow
  base.cand = w.cand; base.cnt = w.cnt; base.thr = d_thresholds; base.cap = static_cast<int32_t>(window_rows);
  set_constraints(base, d_row_filter ? d_row_filter + row_begin / 32 : nullptr,
                  d_row_labels ? d_row_labels + row_begin : nullptr, d_query_labels, label_match);
  rc = run_scan(p, dev, gallery_dtype, base, w.base, padded_queries(n_queries), 0, n_queries, kModeFilter, stream,
                n_rows);
  if (rc != MMRS_OK) return rc;
  MMRS_LAUNCH(launch_range_mark_prefix(w.cand, window_rows, w.cnt, n_queries, w.bitmap, w.word_base, w.chunk_sum,
                                       w.total, dev.sm_count, stream));
  MMRS_CUDA(cudaMemcpyAsync(h_counts, w.total, static_cast<size_t>(n_queries) * sizeof(int64_t),
                            cudaMemcpyDeviceToHost, stream));
  return read_status(w.base.flags, stream);
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
  Carver c(d_workspace);
  const RangeWorkspace w = carve_range(c, window_rows, dim, n_queries);
  MMRS_LAUNCH(launch_range_scatter(w.cand, window_rows, w.cnt, n_queries, w.bitmap, w.word_base, d_out_offsets,
                                   index_offset, d_out_values, d_out_indices, dev.sm_count, stream));
  return MMRS_OK;
}

}  // extern "C"
