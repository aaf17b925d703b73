// range.cu -- finalize of a range search window (mmrs_range_search_window / _scatter in api.cu).
//
// The filter-mode scan appends every key (score, local row) with score >= thr[q] to list q in atomic
// order.  These kernels put each list into ascending row order without a comparison sort: a counting
// sort over a per-(window, query) bitmap in the row-filter word layout (bit r & 31 of word r >> 5).
//   mark     every non-NaN key sets its row's bit
//   count    popcount of each chunk of kRangeChunkWords words
//   prefix   word_base[q][w] = set bits of query q before word w; total[q]
//   scatter  a key's rank = word_base + set bits below it in its word: value and global index land there
// Each (query, row) is appended at most once, so the ranks are a permutation of [0, total[q]) and the
// output does not depend on the append order.
#include "common.cuh"

namespace mmrs {

constexpr int kRangeThreads = 256;
constexpr int kRangeWordsPerThread = 16;
constexpr int64_t kRangeChunkWords = kRangeThreads * kRangeWordsPerThread;   // 4096 words = 131072 rows

// A NaN score's key.  In the scan kernels the compiler builds make_key's `u | 0x80000000` (score >= 0) as a
// float negate (-|x|), which turns a NaN into the canonical NaN 0x7fffffff: the orderable image of -0.0.
// make_key never stores -0.0 (it adds +0.0 first), so that high word is always a NaN score.
__device__ __forceinline__ bool key_is_nan(uint64_t key) {
  const uint32_t o = static_cast<uint32_t>(key >> 32);
  const float s = float_from_orderable(o);
  return o == 0x7fffffffu || s != s;
}

// grid (x, n_queries): block x strides over the keys of list blockIdx.y
__global__ void __launch_bounds__(kRangeThreads) range_mark_kernel(const uint64_t* __restrict__ cand, int64_t cap,
                                                                   const uint32_t* __restrict__ cnt,
                                                                   uint32_t* __restrict__ bitmap, int64_t n_words) {
  const int q = blockIdx.y;
  const int64_t n = cnt[q];
  const uint64_t* list = cand + static_cast<int64_t>(q) * cap;
  uint32_t* bits = bitmap + static_cast<int64_t>(q) * n_words;
  for (int64_t i = blockIdx.x * static_cast<int64_t>(kRangeThreads) + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * kRangeThreads) {
    const uint64_t key = list[i];
    if (key_is_nan(key)) continue;   // `s >= t` is false for a NaN score
    const uint32_t row = key_row(key);
    atomicOr(bits + (row >> 5), 1u << (row & 31));
  }
}

// this thread's kRangeWordsPerThread consecutive words of chunk blockIdx.x of query blockIdx.y
__device__ __forceinline__ void load_words(const uint32_t* bitmap, int64_t n_words, uint32_t (&w)[kRangeWordsPerThread],
                                           int64_t* first) {
  const int64_t w0 = blockIdx.x * kRangeChunkWords + static_cast<int64_t>(threadIdx.x) * kRangeWordsPerThread;
  const uint32_t* src = bitmap + static_cast<int64_t>(blockIdx.y) * n_words + w0;
  *first = w0;
#pragma unroll
  for (int i = 0; i < kRangeWordsPerThread; i += 4) {
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (w0 + i < n_words) v = *reinterpret_cast<const uint4*>(src + i);   // n_words is a multiple of 4
    w[i] = v.x; w[i + 1] = v.y; w[i + 2] = v.z; w[i + 3] = v.w;
  }
}

// sum of `v` over the block (every thread gets it); `excl` = sum over the threads before this one
__device__ __forceinline__ uint32_t block_scan(uint32_t v, uint32_t* excl) {
  __shared__ uint32_t warp_sums[kRangeThreads / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t incl = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t x = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += x;
  }
  if (lane == 31) warp_sums[warp] = incl;
  __syncthreads();
  uint32_t before = 0, total = 0;
#pragma unroll
  for (int i = 0; i < kRangeThreads / 32; ++i) {
    const uint32_t s = warp_sums[i];
    before += i < warp ? s : 0u;
    total += s;
  }
  *excl = before + incl - v;
  return total;
}

// grid (n_chunks, n_queries): chunk_sum[q][c] = set bits of chunk c
__global__ void __launch_bounds__(kRangeThreads) range_count_kernel(const uint32_t* __restrict__ bitmap, int64_t n_words,
                                                                    uint32_t* __restrict__ chunk_sum) {
  uint32_t w[kRangeWordsPerThread];
  int64_t first;
  load_words(bitmap, n_words, w, &first);
  uint32_t s = 0;
#pragma unroll
  for (int i = 0; i < kRangeWordsPerThread; ++i) s += __popc(w[i]);
  uint32_t excl;
  const uint32_t total = block_scan(s, &excl);
  if (threadIdx.x == 0) chunk_sum[static_cast<int64_t>(blockIdx.y) * gridDim.x + blockIdx.x] = total;
}

// grid (n_chunks, n_queries): word_base of every word of chunk c; the last chunk writes total[q]
__global__ void __launch_bounds__(kRangeThreads) range_prefix_kernel(const uint32_t* __restrict__ bitmap, int64_t n_words,
                                                                     const uint32_t* __restrict__ chunk_sum,
                                                                     uint32_t* __restrict__ word_base,
                                                                     int64_t* __restrict__ total) {
  __shared__ uint32_t chunk_base;
  const uint32_t* sums = chunk_sum + static_cast<int64_t>(blockIdx.y) * gridDim.x;
  uint32_t b = 0;
  for (uint32_t c = threadIdx.x; c < blockIdx.x; c += kRangeThreads) b += sums[c];
  uint32_t excl_b;
  const uint32_t base = block_scan(b, &excl_b);
  if (threadIdx.x == 0) chunk_base = base;
  __syncthreads();   // block_scan's shared words are read again below
  uint32_t w[kRangeWordsPerThread];
  int64_t first;
  load_words(bitmap, n_words, w, &first);
  uint32_t s = 0;
#pragma unroll
  for (int i = 0; i < kRangeWordsPerThread; ++i) s += __popc(w[i]);
  uint32_t excl;
  const uint32_t chunk_total = block_scan(s, &excl);
  uint32_t run = chunk_base + excl;
  uint32_t* dst = word_base + static_cast<int64_t>(blockIdx.y) * n_words + first;
#pragma unroll
  for (int i = 0; i < kRangeWordsPerThread; i += 4) {
    uint4 v;
    v.x = run; run += __popc(w[i]);
    v.y = run; run += __popc(w[i + 1]);
    v.z = run; run += __popc(w[i + 2]);
    v.w = run; run += __popc(w[i + 3]);
    if (first + i < n_words) *reinterpret_cast<uint4*>(dst + i) = v;
  }
  if (blockIdx.x == gridDim.x - 1 && threadIdx.x == 0) total[blockIdx.y] = static_cast<int64_t>(chunk_base) + chunk_total;
}

// grid (x, n_queries): every non-NaN key of list q to out[out_off[q] + its rank in row order]
__global__ void __launch_bounds__(kRangeThreads) range_scatter_kernel(
    const uint64_t* __restrict__ cand, int64_t cap, const uint32_t* __restrict__ cnt,
    const uint32_t* __restrict__ bitmap, const uint32_t* __restrict__ word_base, int64_t n_words,
    const int64_t* __restrict__ out_off, int64_t index_offset, float* __restrict__ values,
    int64_t* __restrict__ indices) {
  const int q = blockIdx.y;
  const int64_t n = cnt[q];
  const uint64_t* list = cand + static_cast<int64_t>(q) * cap;
  const uint32_t* bits = bitmap + static_cast<int64_t>(q) * n_words;
  const uint32_t* base = word_base + static_cast<int64_t>(q) * n_words;
  const int64_t off = out_off[q];
  for (int64_t i = blockIdx.x * static_cast<int64_t>(kRangeThreads) + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * kRangeThreads) {
    const uint64_t key = list[i];
    if (key_is_nan(key)) continue;
    const uint32_t row = key_row(key);
    const uint32_t below = bits[row >> 5] & ((1u << (row & 31)) - 1u);
    const int64_t pos = off + base[row >> 5] + __popc(below);
    values[pos] = key_score(key);   // make_key stored -0.0 as +0.0
    indices[pos] = index_offset + row;
  }
}

static int range_list_blocks(int64_t cap, int32_t n_queries, int sm_count) {
  int64_t gx = (cap + kRangeThreads - 1) / kRangeThreads;
  const int64_t most = (8ll * sm_count + n_queries - 1) / n_queries;   // about 8 blocks per SM in all
  if (gx > most) gx = most;
  return static_cast<int>(gx < 1 ? 1 : gx);
}

int64_t range_chunks(int64_t n_words) { return (n_words + kRangeChunkWords - 1) / kRangeChunkWords; }

cudaError_t launch_range_mark_prefix(const uint64_t* cand, int64_t cap, const uint32_t* cnt, int32_t n_queries,
                                     uint32_t* bitmap, uint32_t* word_base, uint32_t* chunk_sum, int64_t* total,
                                     int sm_count, cudaStream_t stream) {
  const int64_t n_words = cap / 32;
  const dim3 lists(range_list_blocks(cap, n_queries, sm_count), n_queries);
  range_mark_kernel<<<lists, kRangeThreads, 0, stream>>>(cand, cap, cnt, bitmap, n_words);
  const dim3 chunks(static_cast<unsigned>(range_chunks(n_words)), n_queries);
  range_count_kernel<<<chunks, kRangeThreads, 0, stream>>>(bitmap, n_words, chunk_sum);
  range_prefix_kernel<<<chunks, kRangeThreads, 0, stream>>>(bitmap, n_words, chunk_sum, word_base, total);
  return cudaGetLastError();
}

cudaError_t launch_range_scatter(const uint64_t* cand, int64_t cap, const uint32_t* cnt, int32_t n_queries,
                                 const uint32_t* bitmap, const uint32_t* word_base, const int64_t* out_off,
                                 int64_t index_offset, float* values, int64_t* indices, int sm_count,
                                 cudaStream_t stream) {
  const dim3 lists(range_list_blocks(cap, n_queries, sm_count), n_queries);
  range_scatter_kernel<<<lists, kRangeThreads, 0, stream>>>(cand, cap, cnt, bitmap, word_base, cap / 32, out_off,
                                                            index_offset, values, indices);
  return cudaGetLastError();
}

}  // namespace mmrs
