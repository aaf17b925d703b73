/*
 * mmrs_b200.h -- C ABI of the B200-native retrieval hot path.
 *
 * The reference (chy980959830/Multi-Modal-Retrieval-System-Image-Search-and-Data-Governance)
 * is pure Python and has no FFI of its own (SURVEY.md section 8b): its "operator
 * interface" for this path is a handful of module-level Python functions.  This
 * header is therefore the boundary a replacement library must export so that the
 * Python mirror of those functions (the package next to this directory) can
 * bind it with ctypes.  Each entry point names the reference expression it
 * replaces (paths relative to the reference checkout):
 *
 *   mmrs_full_scores      code/search_image.py:107   `100. * features.cuda() @ ref_feature.t()`
 *                         CLIP/lab3.py:113-114, CLIP-Chinese/lab_chinese.py:116-117,
 *                         CLIP/union_dataset.py:255-256 (per-class GEMVs, one call)
 *   mmrs_search_topk      code/search_image.py:107 + code/utils.py:17
 *                         `output.topk(k, 1, True, True)` fused, score matrix never stored
 *   mmrs_topk_merge       (new) merge of per-shard top-k after the all-gather
 *   mmrs_selfjoin_pairs(_tc, _stored)  tool/find_repeated_in_same_folder.py:76-95 /
 *                         tool/delete repeated.py:127-135 (pairwise join loop), with the
 *                         predicate cos(e_i, e_j) >= tau named by BASELINE.json
 *   mmrs_threshold_sweep  code/search_image.py:39-79 (eval_threshold / find_thresholds)
 *   mmrs_score_range_batched + mmrs_threshold_sweep_batched
 *                         code/search_image.py:382-389 (the per-class loop of get_similarity :105-117 +
 *                         find_thresholds :58-79) for every class prototype of a batch at once
 *   mmrs_range_search_window + mmrs_range_search_scatter
 *                         code/merge_dataset.py:259-284 `preds = similarity >= threshold`,
 *                         code/union_clip_llava2.py:153-162 (accept every image at or above a class's
 *                         threshold), tool/delete repeated.py (every row within tau of a query) --
 *                         the rows passing a per-query threshold, score matrix never stored
 *   mmrs_resolve_duplicates
 *                         tool/find_repeated_in_same_folder.py:76-95 (the keep / delete walk over the
 *                         similar pairs, in file-size order), on the device
 *
 * Conventions
 *   - every function returns an int status: 0 = ok, negative = error (table below);
 *     nothing throws across the ABI.  mmrs_last_error() returns a thread-local
 *     NUL-terminated description of the most recent failure on the calling thread.
 *   - pointers named d_* are caller-owned DEVICE pointers, h_* are HOST pointers.
 *     The library allocates no persistent device memory: scratch space is a
 *     caller-provided workspace whose size comes from the matching
 *     *_workspace_bytes() query.
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream).
 *     Calls may come from several threads.  Process-global state, all of it
 *     internal and mutex-/atomic-protected: a cache of at most 32 instantiated
 *     CUDA graphs keyed by the caller's workspace pointer (a search replays
 *     the graph captured for its workspace; query / result pointers are
 *     patched into it, they are not part of the key), the launch counter and
 *     the profiling log of the measurement hooks.  Per thread: the error
 *     string, one pinned status word, the device-attribute cache.  Two
 *     searches in flight at the same time need two workspaces.
 *   - matrices are row-major; `ld_*` is the row stride in ELEMENTS.
 *   - there is no CPU fallback: on a device that is not compute capability 10.x
 *     every compute entry point returns MMRS_ERR_ARCH.
 */
#ifndef MMRS_B200_H_
#define MMRS_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default) /* the library itself is built with -fvisibility=hidden */
#endif

#define MMRS_ABI_VERSION 3

/* status codes */
#define MMRS_OK 0
#define MMRS_ERR_ARG (-1)        /* bad argument (shape, alignment, k > n_rows, ...)   */
#define MMRS_ERR_CUDA (-2)       /* a CUDA runtime / driver call failed               */
#define MMRS_ERR_ARCH (-3)       /* device is not sm_100 (B200)                        */
#define MMRS_ERR_WORKSPACE (-4)  /* workspace too small or misaligned                  */
#define MMRS_ERR_ZERO_NORM (-5)  /* normalize_queries=1 and a query row has zero norm
                                    (the reference yields NaN here, search_image.py:157
                                    has no epsilon; we refuse instead)                 */
#define MMRS_ERR_CAPACITY (-6)   /* output capacity too small (self-join pair buffer);
                                    the required count is still reported             */
#define MMRS_ERR_INTERNAL (-7)
#define MMRS_ERR_RETRY (-8)      /* a candidate list overflowed (scores correlated with the tile
                                    stride pattern; rare): the results of this batch are invalid,
                                    repeat it through mmrs_search_topk_exhaustive              */
#define MMRS_ERR_TIMEOUT (-9)    /* fused all-gather: a peer rank did not arrive within
                                    MMRS_GATHER_TIMEOUT_MS (default 20 000)                   */
#define MMRS_ERR_NONFINITE (-10) /* int8 quantisation: a gallery or query row holds a NaN or an infinity */

/* element types of the gallery / embedding matrix */
#define MMRS_DTYPE_F32 0
#define MMRS_DTYPE_BF16 1
#define MMRS_DTYPE_BF16X3 2 /* an fp32 matrix stored as three bf16 planes hi / mid / lo (x == hi + mid + lo,
                               plane stride n_rows * ld elements; mmrs_split_bf16x3 builds it): searched
                               on the tensor cores with six bf16 MMAs per tile and UNROUNDED queries --
                               fp32-mode results (scores within 1e-6) at tensor-core speed */
#define MMRS_DTYPE_I8 3     /* per-row-scaled int8 rows (mmrs_quantize_rows_i8 builds them), see "int8 galleries" */

/*
 * int8 galleries.  Row r is ld bytes: the codes int8[dim] (dim a multiple of 16: zero codes pad the
 * embedding width D up to round_up(D, 16)), then the row's fp32 scale s_r at byte `dim`, then padding;
 * ld >= dim + 16 and ld % 16 == 0 (mmrs_quantize_rows_i8 writes ld = dim + 16).  A row view
 * (gallery + r0 * ld) carries its own scales, so shards and row windows need no second pointer.
 * For ld_gallery, dim and every `ld_*` of an int8 gallery, an element is one byte.
 *
 * Quantisation of a row x (gallery rows on ingest, queries in every search after their optional
 * normalisation): m = max_j |x_j| (fp32), s = fl(m / 127), c_j = clamp(rint(x_j / s), -127, 127) with IEEE
 * division and round half to even; a zero row has s = 0 and zero codes.  A row holding a NaN or an infinity
 * is refused: MMRS_ERR_NONFINITE.
 *
 * Score, on every path (K1, K2, the exhaustive path, full scores, range search):
 *   score(q, r) = fl(fl(float(dot) * a_q) * s_r),   a_q = fl(s_q * scale)
 * where dot = sum_j c_qj * c_rj is the EXACT int32 code dot product; -0.0 is returned as +0.0.  float(dot)
 * is exact for dim <= 1040 (127^2 * 1040 < 2^24) and rounds to nearest above.  The score is a deterministic
 * function of the codes: it does not depend on the path, the tile schedule or the shard count.
 */

/* kernel selection for mmrs_search_topk / mmrs_full_scores */
#define MMRS_PATH_AUTO 0   /* K1 for small batches, K2 (tcgen05) otherwise               */
#define MMRS_PATH_GEMV 1   /* K1: 128-bit streaming + warp-shuffle dot products            */
#define MMRS_PATH_MMA 2    /* K2: TMA + tcgen05.mma, bf16 / bf16x3 / int8 gallery              */

int mmrs_abi_version(void);
const char* mmrs_last_error(void);

/* 0 when `device` is a compute-capability-10.x GPU, MMRS_ERR_ARCH / MMRS_ERR_CUDA otherwise. */
int mmrs_device_check(int device);

/* ---- search: scores ------------------------------------------------------------------- */

/* Scratch bytes needed by mmrs_full_scores. */
size_t mmrs_full_scores_workspace_bytes(int64_t n_rows, int32_t dim, int32_t gallery_dtype,
                                        int32_t n_queries);

/*
 * out[q, i] = scale * <q_q, g_i>     (q_q first divided by its L2 norm when normalize_queries)
 * d_out_scores is [n_queries, ld_out] fp32, ld_out >= n_rows.
 * Replaces code/search_image.py:107 (n_queries == 1, scale == 100, normalize_queries == 0).
 */
int mmrs_full_scores(const void* d_gallery, int64_t n_rows, int32_t dim, int64_t ld_gallery,
                     int32_t gallery_dtype, const float* d_queries, int32_t n_queries,
                     int64_t ld_queries, int32_t normalize_queries, float scale, int32_t path,
                     float* d_out_scores, int64_t ld_out, void* d_workspace,
                     size_t workspace_bytes, void* stream);

/* fp32 [n_rows, ld_src] -> bf16 planes [3, n_rows, ld_dst] (ld_dst % 8 == 0, >= dim; padding zeroed). */
int mmrs_split_bf16x3(const float* d_src, int64_t n_rows, int32_t dim, int64_t ld_src, void* d_dst,
                      int64_t ld_dst, void* stream);

/*
 * Quantise d_src [n_rows, ld_src] (src_dtype MMRS_DTYPE_F32 or MMRS_DTYPE_BF16, `dim` real columns) into int8
 * gallery rows d_dst [n_rows, ld_dst] bytes (see "int8 galleries"): codes [round_up(dim, 16)], zero past dim,
 * the scale at byte round_up(dim, 16), zero up to ld_dst >= round_up(dim, 16) + 16 (ld_dst % 16 == 0).
 * MMRS_ERR_NONFINITE when a row holds a NaN or an infinity (the other rows are still written).
 * Synchronises `stream`.
 */
int mmrs_quantize_rows_i8(const void* d_src, int32_t src_dtype, int64_t n_rows, int32_t dim, int64_t ld_src,
                          void* d_dst, int64_t ld_dst, void* stream);

/* ---- search: fused top-k ------------------------------------------------------------- */

size_t mmrs_search_workspace_bytes(int64_t n_rows, int32_t dim, int32_t gallery_dtype,
                                   int32_t n_queries, int32_t k);

/*
 * Per-query top-k of scale * <q, g_i> over the rows of one gallery shard, returned like
 * torch.topk(k, dim=1, largest=True, sorted=True) (code/utils.py:17): values [n_queries, k]
 * fp32 descending, indices [n_queries, k] int64.  Equal scores are ordered by ascending
 * row index.  index_offset is added to every index (the shard's first global row).
 * gallery_dtype BF16: the query is rounded to bf16 after normalisation (tensor-core mode);
 * F32: everything is fp32.
 * The call synchronises `stream` before returning (it must read back a status word).
 * MMRS_ERR_RETRY: see mmrs_search_topk_exhaustive.
 */
int mmrs_search_topk(const void* d_gallery, int64_t n_rows, int32_t dim, int64_t ld_gallery,
                     int32_t gallery_dtype, const float* d_queries, int32_t n_queries,
                     int64_t ld_queries, int32_t k, int32_t normalize_queries, float scale,
                     int64_t index_offset, int32_t path, float* d_out_values,
                     int64_t* d_out_indices, void* d_workspace, size_t workspace_bytes,
                     void* stream);

/*
 * Same, but the queries come from and the results go to HOST memory (pinned memory makes
 * the copies asynchronous); the gallery stays device-resident.  This is the call shape of
 * the reference's get_similarity(): host tensors in, host numpy out
 * (code/search_image.py:105-109), minus the per-call upload of the whole gallery.
 * The workspace must be mmrs_search_workspace_bytes() + mmrs_search_host_staging_bytes().
 */
size_t mmrs_search_host_staging_bytes(int32_t dim, int32_t n_queries, int32_t k);
int mmrs_search_topk_host(const void* d_gallery, int64_t n_rows, int32_t dim, int64_t ld_gallery,
                          int32_t gallery_dtype, const float* h_queries, int32_t n_queries,
                          int64_t ld_queries, int32_t k, int32_t normalize_queries, float scale,
                          int64_t index_offset, int32_t path, float* h_out_values,
                          int64_t* h_out_indices, void* d_workspace, size_t workspace_bytes,
                          void* stream);

/*
 * Asynchronous forms: enqueue everything on `stream` and return at once, so a caller can keep
 * several batches in flight (the host prepares batch i+1 while the GPU runs batch i).  h_status is
 * one int32 of PINNED host memory owned by the caller and distinct per batch in flight; after the
 * stream (or an event recorded behind the call) has completed, mmrs_search_status(h_status) returns
 * the outcome of that batch -- MMRS_OK, an error, or MMRS_ERR_RETRY.  Results are valid only when
 * it returns MMRS_OK.  One workspace may be shared by consecutive calls on the same stream.
 * d_row_filter, d_row_labels, d_query_labels, label_match restrict the rows a query may return (see
 * "row constraints" below); NULL, NULL, NULL, 0 searches every row.  The same four arguments end the
 * exhaustive, keys and fused-gather searches below.
 */
int mmrs_search_topk_async(const void* d_gallery, int64_t n_rows, int32_t dim, int64_t ld_gallery,
                           int32_t gallery_dtype, const float* d_queries, int32_t n_queries,
                           int64_t ld_queries, int32_t k, int32_t normalize_queries, float scale,
                           int64_t index_offset, int32_t path, float* d_out_values,
                           int64_t* d_out_indices, void* d_workspace, size_t workspace_bytes,
                           int32_t* h_status, const uint32_t* d_row_filter, const int32_t* d_row_labels,
                           const int32_t* d_query_labels, int32_t label_match, void* stream);
int mmrs_search_topk_host_async(const void* d_gallery, int64_t n_rows, int32_t dim,
                                int64_t ld_gallery, int32_t gallery_dtype, const float* h_queries,
                                int32_t n_queries, int64_t ld_queries, int32_t k,
                                int32_t normalize_queries, float scale, int64_t index_offset,
                                int32_t path, float* h_out_values, int64_t* h_out_indices,
                                void* d_workspace, size_t workspace_bytes, int32_t* h_status,
                                const uint32_t* d_row_filter, const int32_t* d_row_labels,
                                const int32_t* d_query_labels, int32_t label_match, void* stream);
int mmrs_search_status(const int32_t* h_status);

/*
 * The exact fallback for a batch that returned MMRS_ERR_RETRY: one query at a time, every row's
 * score becomes a key, one select over all of them (no thresholds, no candidate lists -- cannot
 * overflow).  Needs its own, larger workspace (8 bytes per gallery row: 0.8 GB at 100M rows), which
 * is why it is not part of every search workspace; allocate it for the call and free it again.
 * Synchronises `stream`.
 */
size_t mmrs_search_exhaustive_workspace_bytes(int64_t n_rows, int32_t dim, int32_t n_queries);
int mmrs_search_topk_exhaustive(const void* d_gallery, int64_t n_rows, int32_t dim, int64_t ld_gallery,
                                int32_t gallery_dtype, const float* d_queries, int32_t n_queries,
                                int64_t ld_queries, int32_t k, int32_t normalize_queries, float scale,
                                int64_t index_offset, float* d_out_values, int64_t* d_out_indices,
                                void* d_workspace, size_t workspace_bytes, const uint32_t* d_row_filter,
                                const int32_t* d_row_labels, const int32_t* d_query_labels,
                                int32_t label_match, void* stream);

/*
 * Refined top-k: rescore candidate rows against a full-precision copy of the gallery and keep the k best.
 * d_store [n_rows, ld_store] is that copy (store_dtype MMRS_DTYPE_F32 or MMRS_DTYPE_BF16, dim and ld_store as
 * for a gallery of that dtype); it may live in device memory or in host memory registered with
 * mmrs_host_register (pass the device pointer it returns).  d_queries [n_queries, ld_queries] fp32 (device),
 * d_candidates [n_queries, k_cand] int64 LOCAL rows, -1 = no candidate; the rows of one query must be distinct.
 * The call runs, in stream order: the search's query preparation in the store's dtype (normalisation, bf16
 * rounding for a bf16 store); one score per candidate; the select of the k largest (score, row) keys.
 * Scores: the score of row r for query q is bit for bit mmrs_full_scores(store, path = MMRS_PATH_GEMV)[q, r]
 * (K1's chunk order, fmaf chain and warp reduction; -0.0 returned as +0.0).  Output as mmrs_search_topk:
 * values [n_queries, k] descending, indices + index_offset, equal scores by ascending row; a query with fewer
 * than k candidates is padded with value -inf, index -1.  1 <= k <= min(1024, k_cand).
 * A candidate outside [-1, n_rows) is found on the device and reported as MMRS_ERR_ARG (it is never read).
 * Workspace: mmrs_refine_workspace_bytes(dim, n_queries, k_cand), 256-byte aligned.
 * h_status NULL: the call synchronises `stream` and returns the outcome.  Otherwise h_status is one int32 of
 * pinned host memory: the call returns after enqueueing, and mmrs_search_status(h_status) gives the outcome
 * once the stream has passed the call.
 */
size_t mmrs_refine_workspace_bytes(int32_t dim, int32_t n_queries, int32_t k_cand);
int mmrs_refine_topk(const void* d_store, int32_t store_dtype, int64_t n_rows, int32_t dim, int64_t ld_store,
                     const float* d_queries, int32_t n_queries, int64_t ld_queries, int32_t normalize_queries,
                     float scale, const int64_t* d_candidates, int32_t k_cand, int64_t index_offset, int32_t k,
                     float* d_out_values, int64_t* d_out_indices, void* d_workspace, size_t workspace_bytes,
                     int32_t* h_status, void* stream);

/*
 * Page-lock `bytes` of ordinary host memory at h_ptr (cudaHostRegister, portable and mapped) and return in
 * *d_ptr_out the address kernels read it through: a refine store kept in host memory.  Undo with
 * mmrs_host_unregister(h_ptr) before the memory is freed.
 */
int mmrs_host_register(void* h_ptr, size_t bytes, void** d_ptr_out);
int mmrs_host_unregister(void* h_ptr);

/*
 * Sharded search without a host round trip: each rank writes its local top-k as packed 64-bit keys
 * (order-preserving fp32 score in the high word, ~global_row in the low word; a larger key is a
 * better match and keys are unique), ONE all-gather moves n_queries * k * 8 bytes per rank, and
 * mmrs_topk_merge_keys_async selects the global top-k_out straight from the gathered buffer
 * [n_lists, list_stride] (each list = n_queries * k_in keys, list_stride >= that, in elements).
 * d_out_keys must hold n_queries * k + 1 elements: the LAST one receives the shard's device status
 * word (0 = ok, 1 = candidate-list overflow, ...), so it is gathered along with the keys and every
 * rank can see whether any rank has to repeat the batch.  d_status is one device int32 of scratch,
 * h_status as above.  pad_short == 0: every query must have at least k_out non-zero keys over all lists.
 * pad_short != 0: it may have fewer (the gathered keys of a label-conditioned search), and the missing
 * positions get value -inf, index -1.
 */
int mmrs_search_topk_keys_async(const void* d_gallery, int64_t n_rows, int32_t dim,
                                int64_t ld_gallery, int32_t gallery_dtype, const float* d_queries,
                                int32_t n_queries, int64_t ld_queries, int32_t k,
                                int32_t normalize_queries, float scale, int64_t index_offset,
                                int32_t path, uint64_t* d_out_keys, void* d_workspace,
                                size_t workspace_bytes, int32_t* h_status,
                                const uint32_t* d_row_filter, const int32_t* d_row_labels,
                                const int32_t* d_query_labels, int32_t label_match, void* stream);
int mmrs_topk_merge_keys_async(const uint64_t* d_keys_in, int32_t n_lists, int32_t n_queries,
                               int32_t k_in, int64_t list_stride, int32_t k_out,
                               float* d_out_values, int64_t* d_out_indices, int32_t* d_status,
                               int32_t* h_status, int32_t pad_short, void* stream);

/*
 * Search fused with its all-gather (one process per GPU, NVLink peer memory instead of NCCL):
 * every rank's LAST select stores its top-k_local keys directly into every rank's gather buffer
 * (d_peer_bufs[r] = rank r's buffer, peer-mapped, world * list_stride uint64; rank s owns the
 * slice [s * list_stride, +n_queries * k_local] plus one status word), the last CTA publishes a
 * "ready" flag to every rank with release semantics, a ONE-WARP kernel on each rank waits until all
 * `world` flags carry this call's epoch, and the merge select then writes the global top-k_out --
 * no collective launch, no host round trip, one CUDA graph per call.
 * d_peer_flags[r] = rank r's flag array (2 * world uint32, zero-initialised once): [0, world) ready,
 * [world, 2*world) ack (a rank acks after merging and after it has copied the ranks' status words to
 * private memory; the first kernel of the next call on the slot waits for the acks of the previous
 * epoch before any buffer is overwritten).  d_local_buf / d_local_flags = this rank's own buffer and
 * flag array (local addresses).  The epoch is a counter in the WORKSPACE, bumped on the device by every
 * call: the workspace must be zero-filled once before its first use and belongs to one (shape, stream)
 * slot; calls on a slot are collective -- same order on every rank.  No spinning CTA ever occupies
 * more than one warp, so searches in flight on several streams cannot starve each other.
 * h_status: pinned int32 [world + 2]; after the stream has completed,
 * mmrs_gather_status(h_status, world) is the outcome on every rank alike (MMRS_ERR_RETRY when any
 * rank overflowed; MMRS_ERR_TIMEOUT when a peer never arrived).  n_queries <= 1024, world <= 64,
 * k_local must be the same on every rank and every shard must hold at least k_local rows -- a rank that
 * contributes fewer keys than min(k_out, its rows) can drop rows of the global top-k; callers with shorter
 * shards use the keys variant above and pad.  With a row constraint the merge select pads: fewer than k_out
 * eligible rows over all ranks give -inf / -1.
 */
int mmrs_search_topk_fused_gather_async(
    const void* d_gallery, int64_t n_rows, int32_t dim, int64_t ld_gallery, int32_t gallery_dtype,
    const float* d_queries, int32_t n_queries, int64_t ld_queries, int32_t k_local, int32_t k_out,
    int32_t normalize_queries, float scale, int64_t index_offset, int32_t path,
    uint64_t* const* d_peer_bufs, uint32_t* const* d_peer_flags, uint64_t* d_local_buf,
    uint32_t* d_local_flags, int32_t rank, int32_t world, int64_t list_stride, float* d_out_values,
    int64_t* d_out_indices, void* d_workspace, size_t workspace_bytes, int32_t* h_status,
    const uint32_t* d_row_filter, const int32_t* d_row_labels, const int32_t* d_query_labels,
    int32_t label_match, void* stream);
int mmrs_gather_status(const int32_t* h_status, int32_t world);

/* ---- row constraints ------------------------------------------------------------------- */

/*
 * d_row_filter (NULL = every row) is an allow-list bitmap over the rows of one gallery (shard): uint32
 * words, bit (r & 31) of word (r >> 5) set when local row r may be returned.  PADDING CONTRACT: the array
 * holds at least 4 * ceil(n_rows / 128) words (whole 128-row tiles); bits at or past n_rows are ignored,
 * but those words must be readable.  A shard of a global filter whose first row is a multiple of 128 is
 * the pointer d_words + first_row / 32 (its tail bits belong to the next shard and are ignored).
 *
 * mmrs_pack_row_filter builds one from a device byte mask d_allowed [n_rows] (non-zero = allowed):
 * n_words >= 4 * ceil(n_rows / 128), words past the last row are zeroed; *d_count (device int64)
 * receives the number of allowed rows.  Asynchronous on `stream`.
 */
int mmrs_pack_row_filter(const uint8_t* d_allowed, int64_t n_rows, uint32_t* d_words, int64_t n_words,
                         int64_t* d_count, void* stream);

/* label_match */
#define MMRS_LABEL_SAME 0    /* only rows whose label equals the query's label             */
#define MMRS_LABEL_OTHER 1   /* only rows whose label differs from it (hard negatives)      */

/*
 * d_row_labels (NULL = no label restriction; d_query_labels and label_match are then ignored) is one
 * int32 class id per row of the gallery (shard), each in [0, 2^31 - 1).  PADDING CONTRACT (the
 * bitmap's): the array holds at least 128 * ceil(n_rows / 128) elements (whole 128-row tiles); labels
 * at or past n_rows are never compared, but must be readable.  A shard of a global label array whose
 * first row is a multiple of 128 is the pointer d_row_labels + first_row.  d_query_labels is a DEVICE
 * int32 [n_queries] in every form, the host-I/O one included.  For query q with c = d_query_labels[q]:
 *   c < 0               no label restriction: exactly the unlabeled search of that query;
 *   MMRS_LABEL_SAME     only rows r with d_row_labels[r] == c;
 *   MMRS_LABEL_OTHER    only rows r with d_row_labels[r] != c;
 * and with d_row_filter as well, a row must pass both.
 *
 * A constrained search returns the top-k of an unconstrained one over the eligible rows only (same
 * values, order and tie rule), indices still those of the full gallery (+ index_offset).  k may exceed
 * the eligible rows of a query (a small class, a label absent from the gallery, a shard with few or no
 * allowed rows): that is NOT an error, positions n_eligible .. k-1 get value -inf, index -1 (key 0 in
 * the key outputs, which every merge ignores), so every shard still contributes k entries.
 * A captured graph is keyed on the filter pointer, both label pointers and label_match; the words and
 * labels are read when the search runs, so a caller that rewrites them in place between calls keeps
 * replaying one graph.  NULL, NULL, NULL, 0 gives exactly the graph of the unconstrained search.
 */

/* ---- multi-GPU merge -------------------------------------------------------------------- */

size_t mmrs_topk_merge_workspace_bytes(int32_t n_lists, int32_t n_queries, int32_t k_in);

/*
 * Merge n_lists per-shard results (as gathered by an all-gather: values [n_lists, n_queries,
 * k_in] fp32, indices [n_lists, n_queries, k_in] int64 GLOBAL row ids < 2^32) into the global
 * top-k_out per query with the same order rule (score desc, index asc).
 */
int mmrs_topk_merge(const float* d_values_in, const int64_t* d_indices_in, int32_t n_lists,
                    int32_t n_queries, int32_t k_in, int32_t k_out, float* d_out_values,
                    int64_t* d_out_indices, void* d_workspace, size_t workspace_bytes,
                    void* stream);

/* ---- near-duplicate self-join ---------------------------------------------------------- */

size_t mmrs_selfjoin_workspace_bytes(int64_t n_rows, int32_t dim, int32_t dtype); /* 0: none needed */

/*
 * All pairs (i, j), i < j, row_begin <= i < row_end, with <e_i, e_j> >= threshold, where the
 * rows of d_emb [n_rows, dim] are fp32 (exact mode).  Pairs are written as int64 [count, 2]
 * in UNSPECIFIED order (the Python tier sorts them lexicographically); *d_out_count (device
 * int64) receives the number found even when it exceeds `capacity`
 * (then MMRS_ERR_CAPACITY is returned and only `capacity` pairs are valid).
 * [row_begin, row_end) is this rank's slice of the upper-triangular schedule; any
 * 0 <= row_begin <= row_end <= n_rows is allowed, so consecutive ranges partition the join.
 * The call synchronises `stream`.
 */
int mmrs_selfjoin_pairs(const void* d_emb, int64_t n_rows, int32_t dim, int64_t ld_emb,
                        int32_t dtype, float threshold, int64_t row_begin, int64_t row_end,
                        int64_t* d_out_pairs, int64_t capacity, int64_t* d_out_count,
                        void* d_workspace, size_t workspace_bytes, void* stream);

/*
 * Tensor-core form of the same join: a bf16 tcgen05 pass over d_emb_bf16 (the same rows rounded to
 * bf16) keeps pairs with <e_i, e_j> >= threshold - margin, and every survivor is re-scored in fp32
 * from d_emb_f32 with the arithmetic of mmrs_selfjoin_pairs, so the emitted set is identical to
 * the exact mode's provided margin covers the bf16 rounding and both fp32 accumulations: for rows of
 * norm at most r, margin >= (2^-7 + 2^-16 + dim * 2^-22) * max(1, r^2) (derived in
 * csrc/selfjoin_mma.cu; the Python tier passes exactly this).  The upper triangle is split into panels of 2048 columns dealt round-robin
 * to `world` ranks; this call does rank `rank`'s share.  d_out_count is device int64[2]:
 * [0] pairs found, [1] candidates that passed the prefilter; MMRS_ERR_CAPACITY when either exceeds
 * its capacity (the counts are still reported so the caller can size a retry).
 * Synchronises `stream`.
 */
size_t mmrs_selfjoin_tc_workspace_bytes(int64_t n_rows, int64_t cand_capacity);
int mmrs_selfjoin_pairs_tc(const float* d_emb_f32, int64_t ld_f32, const void* d_emb_bf16,
                           int64_t ld_bf16, int64_t n_rows, int32_t dim, float threshold,
                           float margin, int32_t rank, int32_t world, int64_t* d_out_pairs,
                           int64_t capacity, int64_t* d_out_count, int64_t cand_capacity,
                           void* d_workspace, size_t workspace_bytes, void* stream);

/*
 * The same join on a gallery in its stored format (d_rows as resident: ld_rows in elements for bf16, in bytes
 * for int8), for galleries too large to keep in fp32 next to a copy.  Rank panels, d_out_count [0] pairs /
 * [1] candidates, the capacity protocol and the synchronisation are those of mmrs_selfjoin_pairs_tc.
 *   MMRS_DTYPE_BF16: the tcgen05 pass multiplies the stored values exactly, so the margin only has to cover the
 *     two fp32 accumulations: margin >= dim * 2^-22 * max(1, r^2) for rows of norm at most r
 *     (mmrs_row_norm_range_bf16).  Survivors are re-scored from the same bf16 rows, each element widened to fp32,
 *     with the fmaf chain of mmrs_selfjoin_pairs: the pair set is that join's on the widened rows.
 *   MMRS_DTYPE_I8 (rows as in "int8 galleries", dim <= 131072): tcgen05.mma.kind::i8 gives the exact code product
 *     dot, and the epilogue keeps i < j with fl(fl(float(dot) * s_i) * s_j) >= threshold -- the int8 score with
 *     the lower row as the query at scale 1.  margin must be 0; there is no recheck, candidates are the pairs
 *     (d_out_count[1] == [0]) and cand_capacity is ignored.
 * Any other dtype: MMRS_ERR_ARG.  Replaces tool/find_repeated_in_same_folder.py:76-95's pairwise hash
 * comparison like mmrs_selfjoin_pairs; workspace: mmrs_selfjoin_stored_workspace_bytes(n_rows, dtype,
 * cand_capacity).
 */
size_t mmrs_selfjoin_stored_workspace_bytes(int64_t n_rows, int32_t dtype, int64_t cand_capacity);
int mmrs_selfjoin_pairs_stored(const void* d_rows, int32_t dtype, int64_t ld_rows, int64_t n_rows,
                               int32_t dim, float threshold, float margin, int32_t rank, int32_t world,
                               int64_t* d_out_pairs, int64_t capacity, int64_t* d_out_count,
                               int64_t cand_capacity, void* d_workspace, size_t workspace_bytes,
                               void* stream);

/*
 * Lexicographic (i, j) sort of an int64 [n_pairs, 2] pair list in place -- the order of
 * `triu(S >= tau, 1).nonzero()`.  Row ids must fit 32 bits.  Workspace:
 * mmrs_sort_pairs_workspace_bytes(n_pairs).  Asynchronous on `stream`.
 */
size_t mmrs_sort_pairs_workspace_bytes(int64_t n_pairs);
int mmrs_sort_pairs(int64_t* d_pairs, int64_t n_pairs, void* d_workspace, size_t workspace_bytes,
                    void* stream);

/*
 * d_out_min_max[0 / 1] = smallest / largest L2 norm over the rows of d_emb (fp32).  The tensor-core
 * join's margin bounds the bf16 rounding of UNIT rows; callers scale it by max_norm^2 (or refuse)
 * when rows are not unit-norm.  Asynchronous on `stream`.
 */
int mmrs_row_norm_range(const float* d_emb, int64_t n_rows, int32_t dim, int64_t ld,
                        float* d_out_min_max, void* stream);
/* The same over bf16 rows (d_emb [n_rows, ld] bf16), each element widened to fp32: the margin of the bf16
 * stored-format join.  A row holding a NaN or an infinity makes the max non-finite. */
int mmrs_row_norm_range_bf16(const void* d_emb, int64_t n_rows, int32_t dim, int64_t ld,
                             float* d_out_min_max, void* stream);

/* ---- threshold / F1 sweep (the reference's consumer of the scores) ------------------ */

/*
 * For each of n_thresholds thresholds t: tp = #{pos >= t}, fp = #{neg >= t} over fp32 device
 * score vectors.  d_out_counts is int64 [n_thresholds, 2] = (tp, fp).
 * Replaces the O(T*N) Python `sum(pos_res >= threshold)` loops of
 * code/search_image.py:43-45 inside find_thresholds (:69-70).  Thresholds must be ASCENDING
 * (np.linspace(min, max, 200) is) and n_thresholds <= 4096; they are fp64 like the
 * np.linspace grid of :61; the comparison is done in fp64 as numpy does (fp32 array vs
 * python float promotes the array).
 */
size_t mmrs_threshold_sweep_workspace_bytes(int32_t n_thresholds);
int mmrs_threshold_sweep(const float* d_pos, int64_t n_pos, const float* d_neg, int64_t n_neg,
                         const double* d_thresholds, int32_t n_thresholds,
                         int64_t* d_out_counts, void* d_workspace, size_t workspace_bytes,
                         void* stream);

/* float64 scores (a numpy float64 array compared with the fp64 grid: no rounding on the way in). */
int mmrs_threshold_sweep_f64(const double* d_pos, int64_t n_pos, const double* d_neg, int64_t n_neg,
                             const double* d_thresholds, int32_t n_thresholds,
                             int64_t* d_out_counts, void* d_workspace, size_t workspace_bytes,
                             void* stream);

/*
 * The same sweep without any N-sized host traffic: d_scores [n] fp32 and d_targets [n] int64 stay on
 * the device, positives are the rows with target == label, the threshold grid is
 * np.linspace(min(scores), max(scores), n_thresholds) built on the device exactly as numpy builds it
 * (code/search_image.py:59-61) -- grid_f32 != 0: in float32 as NumPy >= 2 does for float32 scores
 * (NEP 50), grid_f32 == 0: in float64 as NumPy 1.x did -- and returned in d_out_thresholds
 * [n_thresholds] (fp64 either way);
 * d_out_counts as above.  Workspace: mmrs_threshold_sweep_workspace_bytes(n_thresholds) + 256.
 */
int mmrs_threshold_sweep_labeled(const float* d_scores, const int64_t* d_targets, int64_t label,
                                 int64_t n, int32_t n_thresholds, int32_t grid_f32,
                                 double* d_out_thresholds,
                                 int64_t* d_out_counts, void* d_workspace, size_t workspace_bytes,
                                 void* stream);

/*
 * Per-class threshold tuning for a batch of class prototypes (code/search_image.py:382-389: for each
 * class c, get_similarity :105-117 splits the scores by targets == c, find_thresholds :58-79 sweeps a
 * 200-point np.linspace(min, max) grid) with the scores of the whole batch on the device: d_scores is
 * [n_queries, ld_scores] fp32 (e.g. mmrs_full_scores of the prototypes), d_row_filter (nullable) the
 * row-filter bitmap of the gallery (bit r & 31 of word r >> 5 set = row r allowed); a filtered-out row is
 * neither in the range nor counted.
 *
 * mmrs_score_range_batched: each query's order-preserving (min, max) over the allowed rows, -0.0 counted
 * as +0.0 (the key of x is x's bits with the sign bit flipped for x >= 0 and all bits flipped for x < 0).
 * d_range [n_queries, 2] uint32 is ACCUMULATED with min / max, so initialise it to {0xffffffff, 0}; ranges
 * of several row shards combine with a MIN / MAX reduction.  Replaces min(pos_res, neg_res) / max (:59-60).
 *
 * mmrs_threshold_sweep_batched: per query q, the grid np.linspace(min_q, max_q, n_thresholds) of d_range
 * built as mmrs_threshold_sweep_labeled builds it (grid_f32 as there) into d_out_thresholds [n_queries,
 * n_thresholds] fp64, and d_out_counts [n_queries, n_thresholds, 2] int64 = (#pos >= t, #neg >= t) where
 * the positives of q are the allowed rows r with d_row_labels[r] == d_query_labels[q] (int32 each) and
 * the negatives every other allowed row (get_similarity's pos_res / neg_res, :111-116); d_out_n_pos
 * [n_queries] int64 = the positives of q.  Counts and n_pos of several row shards add up when every
 * shard sweeps the same grid (the reduced range).  Workspace:
 * mmrs_threshold_sweep_batched_workspace_bytes(n_queries, n_thresholds).  Both calls are asynchronous on
 * `stream`.
 */
size_t mmrs_threshold_sweep_batched_workspace_bytes(int32_t n_queries, int32_t n_thresholds);
int mmrs_score_range_batched(const float* d_scores, int64_t ld_scores, int32_t n_queries, int64_t n_rows,
                             const uint32_t* d_row_filter, uint32_t* d_range, void* stream);
int mmrs_threshold_sweep_batched(const float* d_scores, int64_t ld_scores, int32_t n_queries, int64_t n_rows,
                                 const int32_t* d_row_labels, const int32_t* d_query_labels,
                                 const uint32_t* d_row_filter, const uint32_t* d_range,
                                 int32_t n_thresholds, int32_t grid_f32, double* d_out_thresholds,
                                 int64_t* d_out_counts, int64_t* d_out_n_pos, void* d_workspace,
                                 size_t workspace_bytes, void* stream);

/*
 * Range search (code/merge_dataset.py:259-284 `preds = similarity >= threshold`): every row r of the gallery
 * with score(q, r) >= d_thresholds[q] (fp32 [n_queries], compared in fp32), where score is the value
 * mmrs_full_scores writes for the same queries, gallery and path.  The rows are processed in windows of
 * `window_rows` rows (a positive multiple of 128, below 2^31) so that the candidate lists are bounded:
 * the workspace holds window_rows 8-byte keys per query
 * (mmrs_range_search_workspace_bytes(window_rows, dim, n_queries); n_queries in [1, 65535]).
 *
 * mmrs_range_search_window: prepares the queries and scans rows [row_begin, min(row_begin + window_rows,
 * n_rows)) (row_begin a multiple of 128; a bf16x3 gallery is passed whole, as to mmrs_full_scores), appends
 * every passing row, and sorts each query's rows by row index.  Blocks until done and writes h_counts
 * [n_queries] int64 (HOST): the matches of each query in this window.  A NaN score never matches.
 * d_row_filter (nullable) is the allow-list bitmap of the whole gallery (mmrs_pack_row_filter);
 * d_row_labels (nullable) / d_query_labels / label_match restrict query q to rows with label ==
 * d_query_labels[q] (MMRS_LABEL_SAME) or != (MMRS_LABEL_OTHER); a negative query label is unrestricted.
 * Status MMRS_ERR_ZERO_NORM as mmrs_full_scores.
 *
 * mmrs_range_search_scatter: writes the window's matches of query q, in ascending row order, to
 * d_out_values / d_out_indices [d_out_offsets[q], d_out_offsets[q] + h_counts[q]) (device int64
 * offsets [n_queries]); an index is index_offset + the row's position inside the window, so pass
 * index_offset = the gallery's global row offset + row_begin.  A -0.0 score is written as +0.0.  Asynchronous on
 * `stream`; the workspace must still hold the preceding window call's state.
 */
size_t mmrs_range_search_workspace_bytes(int64_t window_rows, int32_t dim, int32_t n_queries);
int mmrs_range_search_window(const void* d_gallery, int64_t n_rows, int32_t dim, int64_t ld_gallery,
                             int32_t gallery_dtype, const float* d_queries, int32_t n_queries, int64_t ld_queries,
                             int32_t normalize_queries, float scale, int32_t path, const float* d_thresholds,
                             int64_t row_begin, int64_t window_rows, const uint32_t* d_row_filter,
                             const int32_t* d_row_labels, const int32_t* d_query_labels, int32_t label_match,
                             int64_t* h_counts, void* d_workspace, size_t workspace_bytes, void* stream);
int mmrs_range_search_scatter(int32_t n_queries, int64_t window_rows, int32_t dim, const int64_t* d_out_offsets,
                              int64_t index_offset, float* d_out_values, int64_t* d_out_indices, void* d_workspace,
                              size_t workspace_bytes, void* stream);

/* ---- duplicate resolve: the keep / delete decision on a pair list ------------------------------ */

/*
 * The greedy first-keeper walk of tool/find_repeated_in_same_folder.py:76-95 (for each image in file-size
 * order, `for ref in reference_hashes: if similar: duplicate of ref; break`, else it becomes a reference) on
 * the pairs of the self-join, on the device.  d_pairs is int64 [n_pairs, 2] with ids in [0, n_items), in any
 * order and orientation; repeated pairs and self-pairs are allowed (a self-pair has no effect).  d_order is
 * the walk order: n_order distinct int64 ids in [0, n_items), possibly a subset; null means 0..n_order-1
 * (n_order <= n_items).  d_representative [n_items] int64 receives, for each row v:
 *   v                                          v is kept;
 *   the kept neighbour of v first in d_order   v is removed (a duplicate of that row);
 *   -1                                         v is not in d_order.
 * That is the host walk's result: its representatives are the kept rows in walk order, its duplicates the
 * (row, representative) of the removed rows in walk order.  n_items < 2^31.  A repeated or out-of-range order
 * id and an out-of-range pair id are found on the device and return MMRS_ERR_ARG.
 * h_rounds (HOST int64[2], nullable) receives the rounds run over the worklist of undecided rows and the
 * number of rows the single-warp tail decided (0: the rounds finished alone).
 * Workspace: mmrs_resolve_duplicates_workspace_bytes(n_items, n_order, n_pairs), 256-byte aligned.
 * Synchronises `stream`: it reads the status word and the worklist counts.
 */
size_t mmrs_resolve_duplicates_workspace_bytes(int64_t n_items, int64_t n_order, int64_t n_pairs);
int mmrs_resolve_duplicates(const int64_t* d_pairs, int64_t n_pairs, const int64_t* d_order, int64_t n_order,
                            int64_t n_items, int64_t* d_representative, int64_t* h_rounds, void* d_workspace,
                            size_t workspace_bytes, void* stream);

/* ---- measurement hooks (bench.py; not needed by a product caller) --------------------------- */

/* Number of kernels this library has launched in this process (monotonic). */
int64_t mmrs_launch_count(void);

/* h_out4 = { graph captures, graph replays, replays that re-pointed query/result nodes, captures whose
 * nodes could not be identified for patching } since process start. */
int mmrs_graph_stats(int64_t* h_out4);

/*
 * While enabled, every gallery-scan kernel launch (K1 / K2; the HBM- or tensor-bound kernels) is
 * bracketed by CUDA events on the caller's stream.  mmrs_profile_read() synchronises those events,
 * returns up to `cap` records (oldest first) and clears the log: duration in ms, kind
 * (MMRS_PATH_GEMV or MMRS_PATH_MMA), and the algorithmic gallery bytes the launch streamed
 * (rows visited * dim * element size; int8: rows visited * (dim + 16), the codes and the scale's tail).
 * Returns the number of records written.
 */
int mmrs_profile_enable(int on);
int mmrs_profile_read(float* h_ms, int32_t* h_kind, int64_t* h_bytes, int64_t* h_flops, int32_t cap);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* MMRS_B200_H_ */
