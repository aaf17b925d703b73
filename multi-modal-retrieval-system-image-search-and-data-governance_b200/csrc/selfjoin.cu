// selfjoin.cu -- K5 (exact fp32 mode): thresholded embedding self-join.
//
// The reference's near-duplicate tools compare every image with every kept representative in
// an interpreted double loop (tool/find_repeated_in_same_folder.py:76-95,
// tool/delete repeated.py:127-135).  BASELINE.json replaces the perceptual-hash predicate by
// cos(e_i, e_j) >= tau on unit-norm CLIP embeddings; this kernel evaluates that predicate for
// every pair i < j of an upper-triangular 128x128 block schedule and appends the hits.
//
// Exact mode: fp32 FFMA, k ascending, one accumulator per pair -- the pair set does not depend
// on tile shape or launch geometry.  selfjoin_mma.cu is the tensor-core prefilter whose survivors are
// re-scored with exactly this arithmetic; this kernel serves small inputs and as its cross-check.
//
// The file ends with the extern "C" entry points of its kernels: the exact self-join, the pair sort, the
// row-norm range and the threshold sweeps.
#include <type_traits>

#include "host.h"

namespace mmrs {

constexpr int kSjTile = 128;   // rows of each side per CTA tile
constexpr int kSjBK = 8;       // k-slice staged per iteration
constexpr int kSjThreads = 256;

struct SelfJoinParams {
  const float* emb;
  int64_t n_rows;
  int64_t ld;
  int32_t dim;
  float threshold;
  int64_t row_begin, row_end; // rows of the "i" side owned by this call
  int64_t bi_begin, bi_end;   // the row blocks that hold them
  int64_t nb;                 // number of row blocks
  int64_t total_tiles;
  int64_t* out_pairs;
  int64_t capacity;
  unsigned long long* out_count;
};

// tiles are numbered row-block by row-block: block row bi owns (nb - bi) tiles (bj = bi..nb-1)
__device__ __forceinline__ void decode_tile(int64_t t, int64_t bi0, int64_t nb, int64_t& bi,
                                            int64_t& bj) {
  // tiles before block row b (relative to bi0): f(b) = sum_{x=bi0}^{b-1} (nb - x)
  const double m = static_cast<double>(nb - bi0);
  // solve f(b) <= t: with r = b - bi0, f = r*m - r(r-1)/2
  double r = floor((2.0 * m + 1.0 - sqrt((2.0 * m + 1.0) * (2.0 * m + 1.0) - 8.0 * static_cast<double>(t))) * 0.5);
  int64_t ri = static_cast<int64_t>(r);
  if (ri < 0) ri = 0;
  auto f = [&](int64_t x) { return x * (nb - bi0) - x * (x - 1) / 2; };
  while (ri > 0 && f(ri) > t) --ri;
  while (f(ri + 1) <= t) ++ri;
  bi = bi0 + ri;
  bj = bi + (t - f(ri));
}

__global__ void __launch_bounds__(kSjThreads) selfjoin_f32_kernel(const SelfJoinParams p) {
  __shared__ __align__(16) float As[kSjBK][kSjTile];
  __shared__ __align__(16) float Bs[kSjBK][kSjTile];
  const int tid = threadIdx.x;
  const int ty = tid / 16, tx = tid % 16;
  const int ld_row = tid / 2, ld_k = (tid % 2) * 4;

  for (int64_t t = blockIdx.x; t < p.total_tiles; t += gridDim.x) {
    int64_t bi, bj;
    decode_tile(t, p.bi_begin, p.nb, bi, bj);
    const int64_t i0 = bi * kSjTile, j0 = bj * kSjTile;
    const int64_t arow = min(i0 + ld_row, p.n_rows - 1);
    const int64_t brow = min(j0 + ld_row, p.n_rows - 1);
    const float* ap = p.emb + arow * p.ld + ld_k;
    const float* bp = p.emb + brow * p.ld + ld_k;

    float acc[8][8];
#pragma unroll
    for (int a = 0; a < 8; ++a)
#pragma unroll
      for (int b = 0; b < 8; ++b) acc[a][b] = 0.f;

    for (int k0 = 0; k0 < p.dim; k0 += kSjBK) {
      const float4 av = *reinterpret_cast<const float4*>(ap + k0);
      const float4 bv = *reinterpret_cast<const float4*>(bp + k0);
      __syncthreads();
      As[ld_k + 0][ld_row] = av.x; As[ld_k + 1][ld_row] = av.y;
      As[ld_k + 2][ld_row] = av.z; As[ld_k + 3][ld_row] = av.w;
      Bs[ld_k + 0][ld_row] = bv.x; Bs[ld_k + 1][ld_row] = bv.y;
      Bs[ld_k + 2][ld_row] = bv.z; Bs[ld_k + 3][ld_row] = bv.w;
      __syncthreads();
#pragma unroll
      for (int kk = 0; kk < kSjBK; ++kk) {
        const float4 a0 = *reinterpret_cast<const float4*>(&As[kk][ty * 8]);
        const float4 a1 = *reinterpret_cast<const float4*>(&As[kk][ty * 8 + 4]);
        const float4 b0 = *reinterpret_cast<const float4*>(&Bs[kk][tx * 8]);
        const float4 b1 = *reinterpret_cast<const float4*>(&Bs[kk][tx * 8 + 4]);
        const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
        const float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
        for (int x = 0; x < 8; ++x)
#pragma unroll
          for (int y = 0; y < 8; ++y) acc[x][y] = fmaf(a[x], b[y], acc[x][y]);
      }
    }

#pragma unroll
    for (int x = 0; x < 8; ++x)
#pragma unroll
      for (int y = 0; y < 8; ++y) {
        const int64_t i = i0 + ty * 8 + x, j = j0 + tx * 8 + y;
        if (i >= p.row_begin && i < p.row_end && i < j && j < p.n_rows && acc[x][y] >= p.threshold) {
          const unsigned long long pos = atomicAdd(p.out_count, 1ull);
          if (pos < static_cast<unsigned long long>(p.capacity)) {
            p.out_pairs[2 * pos] = i;
            p.out_pairs[2 * pos + 1] = j;
          }
        }
      }
  }
}

static cudaError_t launch_selfjoin_f32(const float* emb, int64_t n_rows, int32_t dim, int64_t ld,
                                       float threshold, int64_t row_begin, int64_t row_end,
                                       int64_t* out_pairs, int64_t capacity, int64_t* out_count,
                                       int sm_count, cudaStream_t stream) {
  SelfJoinParams p{};
  p.emb = emb; p.n_rows = n_rows; p.ld = ld; p.dim = dim; p.threshold = threshold;
  p.nb = (n_rows + kSjTile - 1) / kSjTile;
  p.row_begin = row_begin; p.row_end = row_end;   // the blocks at either end may hold rows outside the range
  p.bi_begin = row_begin / kSjTile;
  p.bi_end = (row_end + kSjTile - 1) / kSjTile;
  if (p.bi_end > p.nb) p.bi_end = p.nb;
  const int64_t nbi = p.bi_end - p.bi_begin;
  if (nbi <= 0) return cudaSuccess;
  p.total_tiles = nbi * (p.nb - p.bi_begin) - nbi * (nbi - 1) / 2;
  p.out_pairs = out_pairs; p.capacity = capacity;
  p.out_count = reinterpret_cast<unsigned long long*>(out_count);
  int64_t grid = static_cast<int64_t>(sm_count) * 2;
  if (grid > p.total_tiles) grid = p.total_tiles;
  selfjoin_f32_kernel<<<static_cast<int>(grid), kSjThreads, 0, stream>>>(p);
  return cudaGetLastError();
}

// ---- threshold sweep (code/search_image.py:39-79) ------------------------------------------------
// counts[t] = (#pos >= thr_t, #neg >= thr_t) for an ASCENDING threshold grid: each score finds
// how many thresholds it reaches by binary search (fp64 compare, as numpy promotes), bumps one
// histogram bin, and a suffix sum turns the histogram into the counts.
constexpr int kSweepMaxT = 4096;

template <typename S>   // float (numpy float32 scores) or double (float64 scores: no rounding on the way in)
__global__ void __launch_bounds__(256) sweep_hist_kernel(const S* __restrict__ pos, int64_t n_pos,
                                                         const S* __restrict__ neg, int64_t n_neg,
                                                         const double* __restrict__ thr, int32_t n_thr,
                                                         unsigned long long* __restrict__ hist) {
  extern __shared__ double s_thr[];                  // [n_thr]
  uint32_t* s_hist = reinterpret_cast<uint32_t*>(s_thr + n_thr);  // [2][n_thr + 1]
  for (int i = threadIdx.x; i < n_thr; i += blockDim.x) s_thr[i] = thr[i];
  for (int i = threadIdx.x; i < 2 * (n_thr + 1); i += blockDim.x) s_hist[i] = 0;
  __syncthreads();
  const int64_t total = n_pos + n_neg;
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const bool is_neg = i >= n_pos;
    const double x = static_cast<double>(is_neg ? neg[i - n_pos] : pos[i]);
    int lo = 0, hi = n_thr;  // number of thresholds t with x >= t (thresholds ascending)
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (x >= s_thr[mid]) lo = mid + 1; else hi = mid;
    }
    atomicAdd(&s_hist[(is_neg ? n_thr + 1 : 0) + lo], 1u);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * (n_thr + 1); i += blockDim.x)
    if (s_hist[i]) atomicAdd(&hist[i], static_cast<unsigned long long>(s_hist[i]));
}

// ---- fully device-resident variant: scores [Q, ld] + row labels, positives = (label == the query's label) ----
// Per query: min / max of the scores over the allowed rows -> np.linspace(min, max, T) in fp64 exactly as numpy
// builds it (y = arange(T) * step + start with a separately rounded multiply and add, last point = stop) -> the
// same histogram.  Nothing of size N leaves the GPU (code/search_image.py:109 copies all N scores).  One query
// over int64 targets is mmrs_threshold_sweep_labeled; a batch of queries over int32 RowLabels, optionally
// restricted by a row-filter bitmap, is mmrs_threshold_sweep_batched (best_thresholds).
__device__ __forceinline__ uint32_t f2ord(float f) {
  const uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ord2f(uint32_t o) {
  return __uint_as_float((o & 0x80000000u) ? (o & 0x7fffffffu) : ~o);
}
__device__ __forceinline__ bool row_allowed(const uint32_t* __restrict__ filt, int64_t i) {
  return filt == nullptr || ((__ldg(filt + (i >> 5)) >> (i & 31)) & 1u);
}

// Order-preserving (min, max) of each query's scores, -0.0 canonicalised to +0.0 (x + 0.0f), ACCUMULATED into
// range [n_q, 2] with atomicMin / atomicMax (a rank's shard combines with the others' the same way).  A CTA
// covers up to kRangeQG queries of one row range, so a filter word is read once per group of queries.
constexpr int kRangeQG = 8;
__global__ void __launch_bounds__(256) score_range_kernel(const float* __restrict__ scores, int64_t ld, int32_t n_q,
                                                         int64_t n, const uint32_t* __restrict__ filt,
                                                         uint32_t* __restrict__ range) {
  const int n_groups = (n_q + kRangeQG - 1) / kRangeQG;
  for (int g = blockIdx.y; g < n_groups; g += gridDim.y) {
    const int q0 = g * kRangeQG, nqg = min(kRangeQG, n_q - q0);
    uint32_t lo[kRangeQG], hi[kRangeQG];
#pragma unroll
    for (int j = 0; j < kRangeQG; ++j) { lo[j] = 0xffffffffu; hi[j] = 0u; }
    for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n;
         i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
      if (!row_allowed(filt, i)) continue;
#pragma unroll
      for (int j = 0; j < kRangeQG; ++j) {
        if (j < nqg) {
          const uint32_t o = f2ord(scores[(q0 + j) * ld + i] + 0.0f);
          lo[j] = o < lo[j] ? o : lo[j];
          hi[j] = o > hi[j] ? o : hi[j];
        }
      }
    }
#pragma unroll
    for (int j = 0; j < kRangeQG; ++j) {
      if (j < nqg) {
        const uint32_t l = __reduce_min_sync(0xffffffffu, lo[j]);
        const uint32_t h = __reduce_max_sync(0xffffffffu, hi[j]);
        if ((threadIdx.x & 31) == 0 && l <= h) { atomicMin(range + 2 * (q0 + j), l); atomicMax(range + 2 * (q0 + j) + 1, h); }
      }
    }
  }
}

// grid_f32 != 0: NumPy >= 2 semantics (NEP 50): np.linspace of two float32 scalars is computed and
// returned in float32 (delta, step, t * step and + start each rounded to fp32); grid_f32 == 0: NumPy 1.x
// semantics, everything in fp64.  Either way multiply and add are rounded separately (no FMA).
// thr [n_q, n_thr]: row q is the grid of range[q].
__global__ void linspace_kernel(const uint32_t* __restrict__ range, int32_t n_q, int32_t n_thr, int32_t grid_f32,
                                double* __restrict__ thr) {
  const int64_t total = static_cast<int64_t>(n_q) * n_thr;
  for (int64_t idx = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t q = idx / n_thr;
    const int t = static_cast<int>(idx - q * n_thr);
    const float start32 = ord2f(range[2 * q]), stop32 = ord2f(range[2 * q + 1]);
    double v = static_cast<double>(start32);
    if (n_thr > 1) {
      if (t == n_thr - 1) {
        v = static_cast<double>(stop32);
      } else if (grid_f32) {
        const float step = __fdiv_rn(__fsub_rn(stop32, start32), static_cast<float>(n_thr - 1));
        v = static_cast<double>(__fadd_rn(__fmul_rn(static_cast<float>(t), step), start32));
      } else {
        const double start = static_cast<double>(start32), stop = static_cast<double>(stop32);
        const double step = __ddiv_rn(__dsub_rn(stop, start), static_cast<double>(n_thr - 1));
        v = __dadd_rn(__dmul_rn(static_cast<double>(t), step), start);
      }
    }
    thr[idx] = v;
  }
}

// Label sources of the histogram: which rows are positives of query q.
struct TargetsLabel {          // int64 targets, one label for every query (mmrs_threshold_sweep_labeled)
  const int64_t* __restrict__ targets;
  int64_t label;
  __device__ __forceinline__ int64_t row(int64_t i) const { return targets[i]; }
  __device__ __forceinline__ bool positive(int64_t v, int32_t) const { return v == label; }
};
struct RowLabelsSource {       // int32 RowLabels, one label per query (mmrs_threshold_sweep_batched)
  const int32_t* __restrict__ row_labels;
  const int32_t* __restrict__ query_labels;
  __device__ __forceinline__ int32_t row(int64_t i) const { return row_labels[i]; }
  __device__ __forceinline__ bool positive(int32_t v, int32_t query_label) const { return v == query_label; }
};

// Bin of score x in a grid: the number of thresholds t with x >= thr[t], compared in fp64 as numpy does.
// kBinWalk: the grid is non-decreasing with distinct ends -- guess the bin from the linear model of the
// grid and walk to the exact bin against the stored points (the same count as a binary search of a sorted
// grid, in ~2 shared loads instead of log2(T)); kBinFlat: every point equal (min == max, or T == 1);
// kBinSearch: anything else (NaN in the grid) -- the binary search of mmrs_threshold_sweep.
enum : int32_t { kBinSearch = 0, kBinWalk = 1, kBinFlat = 2 };
__device__ __forceinline__ int grid_bin(double x, const double* __restrict__ thr, int32_t n_thr, int32_t mode,
                                        double inv_step) {
  if (mode == kBinFlat) return x >= thr[0] ? n_thr : 0;
  int lo;
  if (mode == kBinWalk) {
    const double d = (x - thr[0]) * inv_step;
    lo = !(d >= 0.0) ? 0 : (d >= static_cast<double>(n_thr) ? n_thr : static_cast<int>(d) + 1);
    if (lo > n_thr) lo = n_thr;
    while (lo > 0 && !(x >= thr[lo - 1])) --lo;
    while (lo < n_thr && x >= thr[lo]) ++lo;
    return lo;
  }
  int hi = n_thr;
  lo = 0;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (x >= thr[mid]) lo = mid + 1; else hi = mid;
  }
  return lo;
}

// hist [n_q, 2, n_thr + 1] (pos bins, then neg bins), ACCUMULATED.  A CTA owns a row range and a group of
// up to `qg` queries whose grids and histograms sit in shared memory, so each row's label and filter word
// are read once per group.  Filtered-out rows are skipped.
template <typename L>
__global__ void __launch_bounds__(512) sweep_hist_labeled_kernel(const float* __restrict__ scores, int64_t ld, int32_t n_q,
                                                                 int64_t n, L src, const uint32_t* __restrict__ filt,
                                                                 const double* __restrict__ thr, int32_t n_thr, int32_t qg,
                                                                 unsigned long long* __restrict__ hist) {
  extern __shared__ double s_thr[];                                    // [qg][n_thr]
  double* s_inv = s_thr + static_cast<size_t>(qg) * n_thr;             // [qg]
  uint32_t* s_hist = reinterpret_cast<uint32_t*>(s_inv + qg);          // [qg][2][n_thr + 1]
  int32_t* s_qlab = reinterpret_cast<int32_t*>(s_hist + static_cast<size_t>(qg) * 2 * (n_thr + 1));   // [qg]
  int32_t* s_mode = s_qlab + qg;                                       // [qg]
  const int hb = 2 * (n_thr + 1);
  const int n_groups = (n_q + qg - 1) / qg;
  for (int g = blockIdx.y; g < n_groups; g += gridDim.y) {
    const int q0 = g * qg, nqg = min(qg, n_q - q0);
    for (int i = threadIdx.x; i < nqg * n_thr; i += blockDim.x) s_thr[i] = thr[static_cast<int64_t>(q0) * n_thr + i];
    for (int i = threadIdx.x; i < nqg * hb; i += blockDim.x) s_hist[i] = 0;
    for (int j = threadIdx.x; j < nqg; j += blockDim.x) {
      s_mode[j] = kBinWalk;
      if constexpr (std::is_same<L, RowLabelsSource>::value) s_qlab[j] = src.query_labels[q0 + j];
      else s_qlab[j] = 0;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < nqg * (n_thr - 1); i += blockDim.x) {
      const int j = i / (n_thr - 1), t = i - j * (n_thr - 1);
      if (!(s_thr[j * n_thr + t] <= s_thr[j * n_thr + t + 1])) s_mode[j] = kBinSearch;
    }
    __syncthreads();
    for (int j = threadIdx.x; j < nqg; j += blockDim.x) {
      const double first = s_thr[j * n_thr], last = s_thr[j * n_thr + n_thr - 1];
      if (s_mode[j] == kBinWalk && first == last) s_mode[j] = kBinFlat;   // non-decreasing with equal ends
      s_inv[j] = s_mode[j] == kBinWalk ? static_cast<double>(n_thr - 1) / (last - first) : 0.0;
    }
    __syncthreads();
    for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n;
         i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
      if (!row_allowed(filt, i)) continue;
      const auto lab = src.row(i);
#pragma unroll 4
      for (int j = 0; j < nqg; ++j) {
        const double x = static_cast<double>(scores[(q0 + j) * ld + i]);
        const int b = grid_bin(x, s_thr + j * n_thr, n_thr, s_mode[j], s_inv[j]);
        atomicAdd(&s_hist[j * hb + (src.positive(lab, s_qlab[j]) ? 0 : n_thr + 1) + b], 1u);
      }
    }
    __syncthreads();
    unsigned long long* h = hist + static_cast<int64_t>(q0) * hb;
    for (int i = threadIdx.x; i < nqg * hb; i += blockDim.x)
      if (s_hist[i]) atomicAdd(&h[i], static_cast<unsigned long long>(s_hist[i]));
    __syncthreads();
  }
}

// One CTA per query, one thread per class (pos / neg): counts[q][t] = sum_{b > t} hist[q][b]; n_pos[q] (when
// non-null) = every positive of the histogram, i.e. the allowed rows of the query's class.
__global__ void sweep_suffix_kernel(const unsigned long long* __restrict__ hist, int32_t n_q, int32_t n_thr,
                                    int64_t* __restrict__ out, int64_t* __restrict__ n_pos) {
  const int c = threadIdx.x;
  if (c >= 2) return;
  for (int64_t q = blockIdx.x; q < n_q; q += gridDim.x) {
    const unsigned long long* h = hist + (q * 2 + c) * (n_thr + 1);
    int64_t* o = out + q * 2 * n_thr;
    unsigned long long run = 0;
    for (int t = n_thr - 1; t >= 0; --t) {
      run += h[t + 1];
      o[2 * t + c] = static_cast<int64_t>(run);
    }
    if (c == 0 && n_pos) n_pos[q] = static_cast<int64_t>(run + h[0]);
  }
}

template <typename S>
static cudaError_t launch_threshold_sweep_t(const S* pos, int64_t n_pos, const S* neg, int64_t n_neg,
                                            const double* thr, int32_t n_thr, int64_t* out_counts,
                                            unsigned long long* hist_ws, int sm_count, cudaStream_t stream) {
  if (n_thr < 1 || n_thr > kSweepMaxT) return cudaErrorInvalidValue;
  cudaError_t e = cudaMemsetAsync(hist_ws, 0, sizeof(unsigned long long) * 2 * (n_thr + 1), stream);
  if (e != cudaSuccess) return e;
  const size_t smem = sizeof(double) * n_thr + sizeof(uint32_t) * 2 * (n_thr + 1);
  const int64_t total = n_pos + n_neg;
  int64_t grid = (total + 256 * 8 - 1) / (256 * 8);
  if (grid > sm_count * 4) grid = sm_count * 4;
  if (grid < 1) grid = 1;
  e = cudaFuncSetAttribute(sweep_hist_kernel<S>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                           static_cast<int>(sizeof(double) * kSweepMaxT + sizeof(uint32_t) * 2 * (kSweepMaxT + 1)));
  if (e != cudaSuccess) return e;
  sweep_hist_kernel<S><<<static_cast<int>(grid), 256, smem, stream>>>(pos, n_pos, neg, n_neg, thr, n_thr, hist_ws);
  e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  sweep_suffix_kernel<<<1, 32, 0, stream>>>(hist_ws, 1, n_thr, out_counts, nullptr);
  return cudaGetLastError();
}

// Shared memory of the labeled histogram: per query its grid, 1 / step, two histograms, its label and bin mode.
static size_t sweep_hist_query_bytes(int32_t n_thr) {
  return sizeof(double) * (n_thr + 1) + sizeof(uint32_t) * 2 * (n_thr + 1) + 2 * sizeof(int32_t);
}
constexpr size_t kSweepHistBudget = 48 << 10;   // four 512-thread CTAs per SM at T <= ~1500 (one query: up to 64 KB)

static cudaError_t launch_score_range(const float* scores, int64_t ld, int32_t n_q, int64_t n, const uint32_t* filt,
                                      uint32_t* range, int sm_count, cudaStream_t stream) {
  const int n_groups = (n_q + kRangeQG - 1) / kRangeQG;
  int64_t gx = (n + 256 * 8 - 1) / (256 * 8);
  const int64_t cap = (static_cast<int64_t>(sm_count) * 4 + n_groups - 1) / n_groups;
  if (gx > cap) gx = cap;
  if (gx < 1) gx = 1;
  score_range_kernel<<<dim3(static_cast<unsigned>(gx), static_cast<unsigned>(n_groups < 65535 ? n_groups : 65535)), 256, 0,
                       stream>>>(scores, ld, n_q, n, filt, range);
  return cudaGetLastError();
}

template <typename L>
static cudaError_t launch_sweep_labeled(const float* scores, int64_t ld, int32_t n_q, int64_t n, L src,
                                        const uint32_t* filt, const uint32_t* range, int32_t n_thr, int32_t grid_f32,
                                        double* thr_out, int64_t* out_counts, int64_t* out_n_pos,
                                        unsigned long long* hist_ws, int sm_count, cudaStream_t stream) {
  cudaError_t e = cudaMemsetAsync(hist_ws, 0, sizeof(unsigned long long) * 2 * (n_thr + 1) * static_cast<size_t>(n_q), stream);
  if (e != cudaSuccess) return e;
  const int64_t total = static_cast<int64_t>(n_q) * n_thr;
  const int64_t lgrid = (total + 255) / 256;
  linspace_kernel<<<static_cast<int>(lgrid < 65535 ? lgrid : 65535), 256, 0, stream>>>(range, n_q, n_thr, grid_f32, thr_out);
  const size_t per_q = sweep_hist_query_bytes(n_thr);
  int32_t qg = static_cast<int32_t>(kSweepHistBudget / per_q);
  if (qg < 1) qg = 1;
  if (qg > n_q) qg = n_q;
  const int n_groups = (n_q + qg - 1) / qg;
  int64_t gx = (n + 512 * 8 - 1) / (512 * 8);
  const int64_t cap = (static_cast<int64_t>(sm_count) * 4 + n_groups - 1) / n_groups;
  if (gx > cap) gx = cap;
  if (gx < 1) gx = 1;
  e = cudaFuncSetAttribute(sweep_hist_labeled_kernel<L>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                           static_cast<int>(sweep_hist_query_bytes(kSweepMaxT) > kSweepHistBudget
                                                ? sweep_hist_query_bytes(kSweepMaxT) : kSweepHistBudget));
  if (e != cudaSuccess) return e;
  sweep_hist_labeled_kernel<L><<<dim3(static_cast<unsigned>(gx), static_cast<unsigned>(n_groups < 65535 ? n_groups : 65535)),
                                 512, per_q * qg, stream>>>(scores, ld, n_q, n, src, filt, thr_out, n_thr, qg, hist_ws);
  sweep_suffix_kernel<<<n_q < 65535 ? n_q : 65535, 32, 0, stream>>>(hist_ws, n_q, n_thr, out_counts, out_n_pos);
  return cudaGetLastError();
}

static cudaError_t launch_threshold_sweep_labeled(const float* scores, const int64_t* targets, int64_t label, int64_t n,
                                                  int32_t n_thr, int32_t grid_f32, double* thr_out, int64_t* out_counts,
                                                  unsigned long long* hist_ws, uint32_t* mm_ws, int sm_count,
                                                  cudaStream_t stream) {
  if (n_thr < 1 || n_thr > kSweepMaxT || n < 1) return cudaErrorInvalidValue;
  cudaError_t e = cudaMemsetAsync(mm_ws, 0xff, sizeof(uint32_t), stream);           // min <- 0xffffffff
  if (e != cudaSuccess) return e;
  e = cudaMemsetAsync(mm_ws + 1, 0, sizeof(uint32_t), stream);                      // max <- 0
  if (e != cudaSuccess) return e;
  e = launch_score_range(scores, n, 1, n, nullptr, mm_ws, sm_count, stream);
  if (e != cudaSuccess) return e;
  return launch_sweep_labeled(scores, n, 1, n, TargetsLabel{targets, label}, nullptr, mm_ws, n_thr, grid_f32, thr_out,
                              out_counts, nullptr, hist_ws, sm_count, stream);
}

static cudaError_t launch_threshold_sweep_batched(const float* scores, int64_t ld, int32_t n_q, int64_t n,
                                                  const int32_t* row_labels, const int32_t* query_labels, const uint32_t* filt,
                                                  const uint32_t* range, int32_t n_thr, int32_t grid_f32, double* thr_out,
                                                  int64_t* out_counts, int64_t* out_n_pos, unsigned long long* hist_ws,
                                                  int sm_count, cudaStream_t stream) {
  if (n_thr < 1 || n_thr > kSweepMaxT || n < 1 || n_q < 1) return cudaErrorInvalidValue;
  return launch_sweep_labeled(scores, ld, n_q, n, RowLabelsSource{row_labels, query_labels}, filt, range, n_thr, grid_f32,
                              thr_out, out_counts, out_n_pos, hist_ws, sm_count, stream);
}

// ---- lexicographic sort of the emitted pairs ----------------------------------------------------------------
// The join kernels append pairs in whatever order their CTAs finish; `triu(S >= tau, 1).nonzero()` of the
// oracle is row-major, i.e. sorted by (i, j).  Pairs are packed into u64 keys (i << 32 | j; row ids fit 32
// bits) and sorted with a bitonic network: sub-sequences of 2048 keys in shared memory, larger strides
// as one pass over global memory each.  O(n log^2 n) -- the pair list is tiny next to the join itself.
constexpr int kSortBlock = 1024;           // threads; one block sorts 2 * kSortBlock keys in shared memory
constexpr int kSortTile = 2 * kSortBlock;

__global__ void pack_pairs_kernel(const int64_t* __restrict__ pairs, int64_t n, uint64_t* __restrict__ keys, int64_t m) {
  const int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (t >= m) return;
  keys[t] = t < n ? (static_cast<uint64_t>(pairs[2 * t]) << 32) | static_cast<uint64_t>(pairs[2 * t + 1] & 0xffffffffll)
                  : ~0ull;   // padding sorts to the end
}
__global__ void unpack_pairs_kernel(const uint64_t* __restrict__ keys, int64_t n, int64_t* __restrict__ pairs) {
  const int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (t >= n) return;
  pairs[2 * t] = static_cast<int64_t>(keys[t] >> 32);
  pairs[2 * t + 1] = static_cast<int64_t>(keys[t] & 0xffffffffull);
}
__device__ __forceinline__ void cmp_swap(uint64_t& a, uint64_t& b, bool ascending) {
  if ((a > b) == ascending) { const uint64_t t = a; a = b; b = t; }
}
// all steps (k, j) with j < kSortTile of the stages k_lo..k_hi for this block's 2048 keys
__global__ void __launch_bounds__(kSortBlock) bitonic_smem_kernel(uint64_t* __restrict__ keys, int64_t k_lo, int64_t k_hi) {
  __shared__ uint64_t s[kSortTile];
  const int64_t base = static_cast<int64_t>(blockIdx.x) * kSortTile;
  s[threadIdx.x] = keys[base + threadIdx.x];
  s[threadIdx.x + kSortBlock] = keys[base + threadIdx.x + kSortBlock];
  __syncthreads();
  for (int64_t k = k_lo; k <= k_hi; k <<= 1) {
    for (int64_t j = (k >> 1) < kSortBlock ? (k >> 1) : kSortBlock; j > 0; j >>= 1) {
      // thread t handles the pair (lo, lo + j) with lo = index whose bit j is clear
      const int64_t t = threadIdx.x;
      const int64_t lo = ((t & ~(j - 1)) << 1) | (t & (j - 1));
      const bool ascending = ((base + lo) & k) == 0;
      cmp_swap(s[lo], s[lo + j], ascending);
      __syncthreads();
    }
  }
  keys[base + threadIdx.x] = s[threadIdx.x];
  keys[base + threadIdx.x + kSortBlock] = s[threadIdx.x + kSortBlock];
}
__global__ void bitonic_global_kernel(uint64_t* __restrict__ keys, int64_t m, int64_t k, int64_t j) {
  const int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (t >= (m >> 1)) return;
  const int64_t lo = ((t & ~(j - 1)) << 1) | (t & (j - 1));
  uint64_t a = keys[lo], b = keys[lo + j];
  const bool ascending = (lo & k) == 0;
  if ((a > b) == ascending) { keys[lo] = b; keys[lo + j] = a; }
}

cudaError_t launch_sort_pairs(int64_t* pairs, int64_t n_pairs, uint64_t* scratch, cudaStream_t stream) {
  if (n_pairs < 2) return cudaSuccess;
  int64_t m = kSortTile;
  while (m < n_pairs) m <<= 1;
  // the workspace holds the power of two >= n_pairs; below one tile only that many keys exist: sort a
  // full tile's worth in shared memory from a smaller buffer by clamping the tile to m0
  int64_t m0 = 1;
  while (m0 < n_pairs) m0 <<= 1;
  if (m0 < kSortTile) {
    // small lists: single-block global passes are enough (at most 11 * 12 / 2 tiny launches)
    pack_pairs_kernel<<<static_cast<int>((m0 + 255) / 256), 256, 0, stream>>>(pairs, n_pairs, scratch, m0);
    for (int64_t k = 2; k <= m0; k <<= 1)
      for (int64_t j = k >> 1; j > 0; j >>= 1)
        bitonic_global_kernel<<<static_cast<int>(((m0 >> 1) + 255) / 256), 256, 0, stream>>>(scratch, m0, k, j);
    unpack_pairs_kernel<<<static_cast<int>((n_pairs + 255) / 256), 256, 0, stream>>>(scratch, n_pairs, pairs);
    return cudaGetLastError();
  }
  m = m0;
  const int tiles = static_cast<int>(m / kSortTile);
  pack_pairs_kernel<<<static_cast<int>((m + 255) / 256), 256, 0, stream>>>(pairs, n_pairs, scratch, m);
  bitonic_smem_kernel<<<tiles, kSortBlock, 0, stream>>>(scratch, 2, kSortTile);
  for (int64_t k = 2 * kSortTile; k <= m; k <<= 1) {
    for (int64_t j = k >> 1; j >= kSortTile; j >>= 1)
      bitonic_global_kernel<<<static_cast<int>(((m >> 1) + 255) / 256), 256, 0, stream>>>(scratch, m, k, j);
    bitonic_smem_kernel<<<tiles, kSortBlock, 0, stream>>>(scratch, k, k);
  }
  unpack_pairs_kernel<<<static_cast<int>((n_pairs + 255) / 256), 256, 0, stream>>>(scratch, n_pairs, pairs);
  return cudaGetLastError();
}

// ---- range of the row norms (guard of the bf16 prefilter margin, which assumes unit rows) -------------------
// T = __nv_bfloat16: the rows of a bf16 gallery, each element widened to fp32 (exactly).  A row holding a NaN or an
// infinity has a NaN or infinite norm, whose bits order above every finite one: the max reports it.
template <typename T>
__global__ void __launch_bounds__(256) row_norm_range_kernel(const T* __restrict__ x, int64_t n_rows, int32_t dim,
                                                             int64_t ld, uint32_t* __restrict__ mm) {
  const int lane = threadIdx.x & 31;
  const int64_t warps = static_cast<int64_t>(gridDim.x) * (blockDim.x >> 5);
  uint32_t lo = 0xffffffffu, hi = 0u;
  for (int64_t r = blockIdx.x * static_cast<int64_t>(blockDim.x >> 5) + (threadIdx.x >> 5); r < n_rows; r += warps) {
    const T* row = x + r * ld;
    float ss = 0.f;
    for (int d = lane; d < dim; d += 32) {
      const float v = static_cast<float>(row[d]);
      ss = fmaf(v, v, ss);
    }
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
    const uint32_t bits = __float_as_uint(sqrtf(ss));     // norms are >= 0: bit order == value order
    lo = bits < lo ? bits : lo;
    hi = bits > hi ? bits : hi;
  }
  if (lane == 0 && lo != 0xffffffffu) { atomicMin(mm, lo); atomicMax(mm + 1, hi); }
}
template <typename T>
static cudaError_t launch_row_norm_range(const T* x, int64_t n_rows, int32_t dim, int64_t ld, float* out_min_max,
                                         int sm_count, cudaStream_t stream) {
  uint32_t* mm = reinterpret_cast<uint32_t*>(out_min_max);
  cudaError_t e = cudaMemsetAsync(mm, 0xff, sizeof(uint32_t), stream);
  if (e != cudaSuccess) return e;
  e = cudaMemsetAsync(mm + 1, 0, sizeof(uint32_t), stream);
  if (e != cudaSuccess) return e;
  int64_t grid = (n_rows + 7) / 8;
  if (grid > static_cast<int64_t>(sm_count) * 8) grid = static_cast<int64_t>(sm_count) * 8;
  row_norm_range_kernel<T><<<static_cast<int>(grid), 256, 0, stream>>>(x, n_rows, dim, ld, mm);
  return cudaGetLastError();
}


// ---- host side: the entry points --------------------------------------------------------------------------------
// The sweeps' histograms: two [n_thresholds + 1] counter arrays per query.  The labeled sweep keeps the bits of the
// score range it bins in front of them.
struct SweepWorkspace {
  uint32_t* range;             // [2] min, max score (order-preserving bits); labeled sweep only
  unsigned long long* hist;    // [n_queries, 2, n_thresholds + 1]
};

static SweepWorkspace carve_sweep(Carver& c, int32_t n_queries, int32_t n_thresholds, bool with_range) {
  SweepWorkspace w{};
  if (with_range) w.range = c.take<uint32_t>(2 * sizeof(uint32_t));
  w.hist = c.take<unsigned long long>(sizeof(unsigned long long) * 2 * (static_cast<size_t>(n_thresholds) + 1) *
                                      n_queries);
  return w;
}

// mmrs_threshold_sweep (fp32 scores) and mmrs_threshold_sweep_f64
template <typename S>
static int threshold_sweep(const S* d_pos, int64_t n_pos, const S* d_neg, int64_t n_neg, const double* d_thresholds,
                           int32_t n_thresholds, int64_t* d_out_counts, void* d_workspace, size_t workspace_bytes,
                           void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceInfo dev;
  int rc = current_device(&dev);
  if (rc != MMRS_OK) return rc;
  if (n_thresholds < 1 || n_thresholds > 4096) return fail(MMRS_ERR_ARG, "n_thresholds must be in [1, 4096]");
  if (n_pos < 0 || n_neg < 0 || (n_pos > 0 && !d_pos) || (n_neg > 0 && !d_neg) || !d_thresholds || !d_out_counts)
    return fail(MMRS_ERR_ARG, "bad arguments");
  rc = check_workspace(d_workspace, workspace_bytes, mmrs_threshold_sweep_workspace_bytes(n_thresholds),
                       /*aligned=*/false);
  if (rc != MMRS_OK) return rc;
  Carver c(d_workspace);
  const SweepWorkspace w = carve_sweep(c, 1, n_thresholds, false);
  MMRS_LAUNCH(launch_threshold_sweep_t<S>(d_pos, n_pos, d_neg, n_neg, d_thresholds, n_thresholds, d_out_counts, w.hist,
                                          dev.sm_count, stream));
  return MMRS_OK;
}

}  // namespace mmrs

using namespace mmrs;

extern "C" {

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
  if (row_begin < 0 || row_end > n_rows || row_begin > row_end)
    return fail(MMRS_ERR_ARG, "row range [%lld, %lld) invalid", (long long)row_begin, (long long)row_end);
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
  rc = check_workspace(d_workspace, workspace_bytes, mmrs_sort_pairs_workspace_bytes(n_pairs), /*aligned=*/false);
  if (rc != MMRS_OK) return rc;
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

int mmrs_row_norm_range_bf16(const void* d_emb, int64_t n_rows, int32_t dim, int64_t ld, float* d_out_min_max,
                             void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceInfo dev;
  int rc = current_device(&dev);
  if (rc != MMRS_OK) return rc;
  if (!d_emb || !d_out_min_max || n_rows < 1 || dim < 1 || ld < dim) return fail(MMRS_ERR_ARG, "bad arguments");
  MMRS_LAUNCH(launch_row_norm_range(static_cast<const __nv_bfloat16*>(d_emb), n_rows, dim, ld, d_out_min_max,
                                    dev.sm_count, stream));
  return MMRS_OK;
}

size_t mmrs_threshold_sweep_workspace_bytes(int32_t n_thresholds) {
  if (n_thresholds < 1) n_thresholds = 1;
  Carver c(nullptr);
  carve_sweep(c, 1, n_thresholds, false);
  return c.off;
}

int mmrs_threshold_sweep(const float* d_pos, int64_t n_pos, const float* d_neg, int64_t n_neg,
                         const double* d_thresholds, int32_t n_thresholds, int64_t* d_out_counts,
                         void* d_workspace, size_t workspace_bytes, void* stream) {
  return threshold_sweep(d_pos, n_pos, d_neg, n_neg, d_thresholds, n_thresholds, d_out_counts, d_workspace,
                         workspace_bytes, stream);
}

int mmrs_threshold_sweep_f64(const double* d_pos, int64_t n_pos, const double* d_neg, int64_t n_neg,
                             const double* d_thresholds, int32_t n_thresholds, int64_t* d_out_counts,
                             void* d_workspace, size_t workspace_bytes, void* stream) {
  return threshold_sweep(d_pos, n_pos, d_neg, n_neg, d_thresholds, n_thresholds, d_out_counts, d_workspace,
                         workspace_bytes, stream);
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
  Carver sizing(nullptr);
  carve_sweep(sizing, 1, n_thresholds, true);   // mmrs_threshold_sweep_workspace_bytes + 256
  rc = check_workspace(d_workspace, workspace_bytes, sizing.off, /*aligned=*/false);
  if (rc != MMRS_OK) return rc;
  Carver c(d_workspace);
  const SweepWorkspace w = carve_sweep(c, 1, n_thresholds, true);
  MMRS_LAUNCH(launch_threshold_sweep_labeled(d_scores, d_targets, label, n, n_thresholds, grid_f32, d_out_thresholds,
                                             d_out_counts, w.hist, w.range, dev.sm_count, stream));
  return MMRS_OK;
}

size_t mmrs_threshold_sweep_batched_workspace_bytes(int32_t n_queries, int32_t n_thresholds) {
  if (n_queries < 1) n_queries = 1;
  if (n_thresholds < 1) n_thresholds = 1;
  Carver c(nullptr);
  carve_sweep(c, n_queries, n_thresholds, false);
  return c.off;
}

int mmrs_score_range_batched(const float* d_scores, int64_t ld_scores, int32_t n_queries, int64_t n_rows,
                             const uint32_t* d_row_filter, uint32_t* d_range, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceInfo dev;
  int rc = current_device(&dev);
  if (rc != MMRS_OK) return rc;
  if (n_queries == 0 || n_rows == 0) return MMRS_OK;
  if (n_queries < 0 || n_rows < 0 || ld_scores < n_rows || !d_scores || !d_range) return fail(MMRS_ERR_ARG, "bad arguments");
  MMRS_LAUNCH(launch_score_range(d_scores, ld_scores, n_queries, n_rows, d_row_filter, d_range, dev.sm_count, stream));
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
  rc = check_workspace(d_workspace, workspace_bytes, mmrs_threshold_sweep_batched_workspace_bytes(n_queries, n_thresholds),
                       /*aligned=*/false);
  if (rc != MMRS_OK) return rc;
  Carver c(d_workspace);
  const SweepWorkspace w = carve_sweep(c, n_queries, n_thresholds, false);
  MMRS_LAUNCH(launch_threshold_sweep_batched(d_scores, ld_scores, n_queries, n_rows, d_row_labels, d_query_labels,
                                             d_row_filter, d_range, n_thresholds, grid_f32, d_out_thresholds,
                                             d_out_counts, d_out_n_pos, w.hist, dev.sm_count, stream));
  return MMRS_OK;
}

}  // extern "C"
