// scan_gemv.cu -- K1: bandwidth-bound small-batch scan.
//
// Replaces the reference's `features.cuda() @ ref_feature.t()` (code/search_image.py:107) for
// 1..8 queries per pass: every warp streams R gallery rows with coalesced 128-bit
// L1-bypassing loads (one 512-byte row segment per load instruction), multiplies them with
// the query chunk it holds in shared memory, and finishes the R x QN dot products with one
// transposing warp-shuffle reduction (31 shuffles for 32 sums instead of 160).  The epilogue
// never stores the score matrix unless asked to (kModeScores): it either seeds a dense key list
// (kModeDense) or appends the keys that pass the running k-th-best bound (kModeFilter).
//
// HBM roofline: N*D*sizeof(T) bytes per pass (SURVEY.md section 8d).  The FP32 pipe allows about
// 11.5 bf16 elements/clk/SM at 6.5 TB/s, i.e. QN <= 4 keeps the kernel memory-bound; larger
// batches belong to K2 (scan_mma.cu).
#include "common.cuh"

namespace mmrs {

template <typename T> struct Chunk;
template <> struct Chunk<__nv_bfloat16> {
  static constexpr int CH = 8;  // elements per 16-byte load
  static __device__ __forceinline__ void unpack(const uint4& g, float (&f)[8]) {
    f[0] = __uint_as_float(g.x << 16); f[1] = __uint_as_float(g.x & 0xffff0000u);
    f[2] = __uint_as_float(g.y << 16); f[3] = __uint_as_float(g.y & 0xffff0000u);
    f[4] = __uint_as_float(g.z << 16); f[5] = __uint_as_float(g.z & 0xffff0000u);
    f[6] = __uint_as_float(g.w << 16); f[7] = __uint_as_float(g.w & 0xffff0000u);
  }
};
template <> struct Chunk<float> {
  static constexpr int CH = 4;
  static __device__ __forceinline__ void unpack(const uint4& g, float (&f)[4]) {
    f[0] = __uint_as_float(g.x); f[1] = __uint_as_float(g.y);
    f[2] = __uint_as_float(g.z); f[3] = __uint_as_float(g.w);
  }
};

// Sum V per-lane partials across the warp.  While more than one value is live each stage
// halves the set (lanes with bit `O` keep the upper half), afterwards it is a plain butterfly.
// On return lane l holds the total of value index l / (32 / V).
template <int N, int O>
struct TransposeReduce {
  static __device__ __forceinline__ void run(float* v, int lane) {
    if constexpr (N > 1) {
      const bool up = (lane & O) != 0;
#pragma unroll
      for (int i = 0; i < N / 2; ++i) {
        const float send = up ? v[i] : v[i + N / 2];
        const float keep = up ? v[i + N / 2] : v[i];
        v[i] = keep + __shfl_xor_sync(0xffffffffu, send, O);
      }
      if constexpr (O > 1) TransposeReduce<N / 2, O / 2>::run(v, lane);
    } else {
      v[0] += __shfl_xor_sync(0xffffffffu, v[0], O);
      if constexpr (O > 1) TransposeReduce<1, O / 2>::run(v, lane);
    }
  }
};

constexpr int kGemvThreads = 256;
constexpr int kGemvWarps = kGemvThreads / 32;

// LABELED: label-conditioned search (p.row_labels != nullptr, dense / filter modes only).  A separate
// instantiation, so that the unlabeled kernels keep their code and registers.
template <typename T, int QN, int R, int MODE, bool LABELED = false>
__global__ void __launch_bounds__(kGemvThreads, 2) scan_gemv_kernel(const ScanParams p) {
  constexpr int CH = Chunk<T>::CH;
  constexpr int H = CH / 4;  // float4 pieces of a query chunk
  constexpr int V = QN * R;
  static_assert(V <= 32 && (V & (V - 1)) == 0, "R*QN must be a power of two <= 32");
  static_assert(kTileRows % (kGemvWarps * R) == 0, "tile must split evenly over the warps");

  // Query chunks, laid out [QN][H][n_chunks] in float4 so that consecutive lanes read
  // consecutive 16-byte words (conflict-free LDS.128).
  extern __shared__ float4 q_smem[];
  const int n_chunks = p.dim / CH;
  pdl_launch_dependents();
  pdl_wait();   // queries (prep kernel) and thresholds (previous select) come from predecessors
  for (int i = threadIdx.x; i < QN * H * n_chunks; i += kGemvThreads) {
    const int c = i % n_chunks;
    const int h = (i / n_chunks) % H;
    const int qi = i / (n_chunks * H);
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (qi < p.nq)
      v = *reinterpret_cast<const float4*>(p.queries + static_cast<size_t>(p.q0 + qi) * p.ldq +
                                           c * CH + h * 4);
    q_smem[i] = v;
  }
  __syncthreads();

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int REP = 32 / V;
  const int my_val = lane / REP;          // which of the V sums this lane ends up owning
  const int my_r = my_val / QN, my_q = my_val % QN;
  const bool owner = (lane % REP) == 0 && my_q < p.nq;

  float my_thr = 0.f;
  if constexpr (MODE == kModeFilter) {
    if (owner) my_thr = p.thr[p.q0 + my_q];
  }
  int32_t my_label = -1;   // label-conditioned search: the owned query's label (< 0: no restriction)
  if constexpr (LABELED) {
    if (owner) my_label = __ldg(p.query_labels + p.q0 + my_q);
  }

  const T* __restrict__ gal = static_cast<const T*>(p.gallery);
  const int64_t last_row = p.n_rows - 1;

  for (int j = blockIdx.x; j < p.sched.n_sel; j += gridDim.x) {
    const int t = j * p.sched.tile_inc;
    if (p.sched.tile_exc != 0 && (t % p.sched.tile_exc) == 0) continue;
    const int64_t tile_row0 = static_cast<int64_t>(t) * kTileRows;

#pragma unroll 1
    for (int it = 0; it < kTileRows / (kGemvWarps * R); ++it) {
      const int64_t row0 = tile_row0 + it * (kGemvWarps * R) + warp * R;
      if constexpr (MODE != kModeDense) {
        if (row0 > last_row) break;  // warp-uniform; dense mode still has to zero its slots
      }
      const T* rp[R];
#pragma unroll
      for (int r = 0; r < R; ++r) {
        const int64_t row = row0 + r;
        rp[r] = gal + (row <= last_row ? row : last_row) * p.ld;  // clamp: tail rows re-read the last row
      }
      float acc[R][QN];
#pragma unroll
      for (int r = 0; r < R; ++r)
#pragma unroll
        for (int qi = 0; qi < QN; ++qi) acc[r][qi] = 0.f;

      for (int c = lane; c < n_chunks; c += 32) {
        uint4 g[R];
#pragma unroll
        for (int r = 0; r < R; ++r) g[r] = ldg_stream_16B(rp[r] + c * CH);
        float qv[QN][CH];
#pragma unroll
        for (int qi = 0; qi < QN; ++qi)
#pragma unroll
          for (int h = 0; h < H; ++h) {
            const float4 x = q_smem[(qi * H + h) * n_chunks + c];
            qv[qi][h * 4 + 0] = x.x; qv[qi][h * 4 + 1] = x.y;
            qv[qi][h * 4 + 2] = x.z; qv[qi][h * 4 + 3] = x.w;
          }
#pragma unroll
        for (int r = 0; r < R; ++r) {
          float f[CH];
          Chunk<T>::unpack(g[r], f);
#pragma unroll
          for (int qi = 0; qi < QN; ++qi)
#pragma unroll
            for (int e = 0; e < CH; ++e) acc[r][qi] = fmaf(f[e], qv[qi][e], acc[r][qi]);
        }
      }

      float v[V];
#pragma unroll
      for (int r = 0; r < R; ++r)
#pragma unroll
        for (int qi = 0; qi < QN; ++qi) v[r * QN + qi] = acc[r][qi];
      TransposeReduce<V, 16>::run(v, lane);

      if (owner) {
        const int64_t row = row0 + my_r;
        const float s = v[0] * p.scale;
        const int q = p.q0 + my_q;
        // the bitmap covers whole tiles, so the word of a tail row past last_row is readable (and zero)
        bool row_ok = row <= last_row;
        if constexpr (MODE != kModeScores) {
          if (p.row_filter != nullptr) row_ok = row_ok && row_allowed(__ldg(p.row_filter + (row >> 5)), row);
          // the labels cover whole tiles too
          if constexpr (LABELED) {
            if (my_label >= 0) row_ok = row_ok && label_ok(__ldg(p.row_labels + row), my_label, p.label_match);
          }
        }
        if constexpr (MODE == kModeScores) {
          if (row_ok) p.out_scores[static_cast<int64_t>(q) * p.ld_out + row] = s;
        } else if constexpr (MODE == kModeDense) {
          const int64_t slot = static_cast<int64_t>(j) * kTileRows + (row - tile_row0);
          p.cand[static_cast<int64_t>(q) * p.cap + slot] =
              row_ok ? make_key(s, static_cast<uint32_t>(row)) : 0ull;
        } else {
          if (row_ok && !(s < my_thr)) {
            const uint32_t pos = atomicAdd(p.cnt + q, 1u);
            if (pos < static_cast<uint32_t>(p.cap))
              p.cand[static_cast<int64_t>(q) * p.cap + pos] = make_key(s, static_cast<uint32_t>(row));
          }
        }
      }
    }
  }
}

template <typename T, int QN, int R>
static cudaError_t launch_gemv_mode(const ScanParams& p, int mode, int sm_count,
                                    cudaStream_t stream) {
  const size_t smem = static_cast<size_t>(QN) * p.dim * sizeof(float);
  auto go = [&](auto kernel) -> cudaError_t {
    cudaError_t e = cudaSuccess;
    if (smem > 48 * 1024) {
      e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               static_cast<int>(smem));
      if (e != cudaSuccess) return e;
    }
    int occ = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, kGemvThreads, smem);
    if (e != cudaSuccess) return e;
    if (occ < 1) occ = 1;
    int grid = sm_count * occ;
    if (grid > p.sched.n_sel) grid = p.sched.n_sel;
    if (grid < 1) grid = 1;
    return launch_pdl(kernel, dim3(grid), dim3(kGemvThreads), smem, stream, p);
  };
  const bool labeled = p.row_labels != nullptr;
  switch (mode) {
    case kModeScores: return go(scan_gemv_kernel<T, QN, R, kModeScores>);
    case kModeDense:
      return labeled ? go(scan_gemv_kernel<T, QN, R, kModeDense, true>) : go(scan_gemv_kernel<T, QN, R, kModeDense>);
    default:
      return labeled ? go(scan_gemv_kernel<T, QN, R, kModeFilter, true>) : go(scan_gemv_kernel<T, QN, R, kModeFilter>);
  }
}

template <typename T>
static cudaError_t launch_gemv_q(const ScanParams& p, int mode, int sm_count, cudaStream_t stream) {
  if (p.nq <= 1) return launch_gemv_mode<T, 1, 8>(p, mode, sm_count, stream);
  if (p.nq <= 2) return launch_gemv_mode<T, 2, 8>(p, mode, sm_count, stream);
  if (p.nq <= 4) return launch_gemv_mode<T, 4, 8>(p, mode, sm_count, stream);
  return launch_gemv_mode<T, 8, 4>(p, mode, sm_count, stream);
}

cudaError_t launch_scan_gemv(const ScanParams& p, int32_t dtype, int mode, int sm_count,
                             cudaStream_t stream) {
  if (p.nq < 1 || p.nq > 8) return cudaErrorInvalidValue;
  if (dtype == MMRS_DTYPE_BF16) return launch_gemv_q<__nv_bfloat16>(p, mode, sm_count, stream);
  return launch_gemv_q<float>(p, mode, sm_count, stream);
}

// ---- query preparation ------------------------------------------------------------------------
// One warp per query row: optional L2 normalisation `x / x.norm()` (the reference idiom,
// code/search_image.py:157 -- sqrt of the fp32 sum of squares, true division, no epsilon),
// optional rounding to bf16 (tensor-core mode), zero padding to [n_rows_padded, ld_out].
__global__ void __launch_bounds__(256) prep_queries_kernel(
    const float* __restrict__ q, int32_t n_queries, int64_t ldq, int32_t dim, int32_t normalize,
    int32_t round_bf16, float* __restrict__ out_f32, __nv_bfloat16* __restrict__ out_bf16,
    int32_t n_rows_padded, int32_t ld_out, int32_t* flags, const GatherPrologue gp) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  pdl_launch_dependents();
  pdl_wait();   // the previous search on this stream may still be reading the prepared queries
  if (gp.epoch != nullptr && blockIdx.x == 0 && threadIdx.x == 0) {
    // fused all-gather: this call's sequence number on its slot (the same on every rank, calls are
    // collective), and the guarantee that every rank has finished merging the previous use of the
    // slot's gather buffers before this call's producer select overwrites them
    const uint32_t epoch = *gp.epoch + 1u;
    *gp.epoch = epoch;
    wait_all_ge(gp.ack_flags, gp.world, epoch - 1u, flags, gp.timeout_ns);
  }
  if (row >= n_rows_padded) return;
  float inv_den = 1.f;
  const bool real = row < n_queries;
  const float* src = q + static_cast<int64_t>(row) * ldq;
  if (real && normalize) {
    float ss = 0.f;
    for (int d = lane; d < dim; d += 32) ss = fmaf(src[d], src[d], ss);
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
    inv_den = sqrtf(ss);
    if (!(inv_den > 0.f) && lane == 0) atomicOr(flags, kFlagZeroNorm);
  }
  for (int d = lane; d < ld_out; d += 32) {
    float v = 0.f;
    if (real && d < dim) v = normalize ? src[d] / inv_den : src[d];
    if (round_bf16 == 1) {
      const __nv_bfloat16 b = __float2bfloat16_rn(v);
      v = __bfloat162float(b);
      if (out_bf16) out_bf16[static_cast<int64_t>(row) * ld_out + d] = b;
    } else if (round_bf16 == 2 && out_bf16) {
      // fp32 emulation on tensor cores: three planes hi / mid / lo with v == hi + mid + lo
      const int64_t plane = static_cast<int64_t>(n_rows_padded) * ld_out;
      const __nv_bfloat16 hi = __float2bfloat16_rn(v);
      const float r1 = v - __bfloat162float(hi);
      const __nv_bfloat16 mid = __float2bfloat16_rn(r1);
      const __nv_bfloat16 lo = __float2bfloat16_rn(r1 - __bfloat162float(mid));
      const int64_t o = static_cast<int64_t>(row) * ld_out + d;
      out_bf16[o] = hi; out_bf16[o + plane] = mid; out_bf16[o + 2 * plane] = lo;
    }
    out_f32[static_cast<int64_t>(row) * ld_out + d] = v;
  }
}

cudaError_t launch_prep_queries(const float* q, int32_t n_queries, int64_t ldq, int32_t dim,
                                int32_t normalize, int32_t round_bf16, float* out_f32,
                                __nv_bfloat16* out_bf16, int32_t n_rows_padded, int32_t ld_out,
                                int32_t* flags, const GatherPrologue& gp, cudaStream_t stream) {
  const int warps_per_block = 8;
  const int grid = (n_rows_padded + warps_per_block - 1) / warps_per_block;
  return launch_pdl(prep_queries_kernel, dim3(grid), dim3(warps_per_block * 32), 0, stream, q, n_queries,
                    ldq, dim, normalize, round_bf16, out_f32, out_bf16, n_rows_padded, ld_out, flags, gp);
}
const void* prep_kernel_handle() { return reinterpret_cast<const void*>(prep_queries_kernel); }
static_assert(kPrepKernelParams == 12, "api.cu patches parameter 0 of a kPrepKernelParams-parameter kernel");

// ---- fp32 -> three bf16 planes (gallery ingest for the fp32 tensor-core path) ------------------------
__global__ void __launch_bounds__(256) split_bf16x3_kernel(const float* __restrict__ src, int64_t n_rows, int32_t dim,
                                                           int64_t ld_src, __nv_bfloat16* __restrict__ dst, int64_t ld_dst) {
  const int64_t total = n_rows * ld_dst;
  const int64_t plane = n_rows * ld_dst;
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t r = i / ld_dst;
    const int32_t d = static_cast<int32_t>(i % ld_dst);
    const float v = d < dim ? src[r * ld_src + d] : 0.f;
    const __nv_bfloat16 hi = __float2bfloat16_rn(v);
    const float r1 = v - __bfloat162float(hi);
    const __nv_bfloat16 mid = __float2bfloat16_rn(r1);
    const __nv_bfloat16 lo = __float2bfloat16_rn(r1 - __bfloat162float(mid));
    dst[i] = hi; dst[i + plane] = mid; dst[i + 2 * plane] = lo;
  }
}
cudaError_t launch_split_bf16x3(const float* src, int64_t n_rows, int32_t dim, int64_t ld_src, __nv_bfloat16* dst,
                                int64_t ld_dst, int sm_count, cudaStream_t stream) {
  if (n_rows <= 0) return cudaSuccess;
  int64_t grid = (n_rows * ld_dst + 255) / 256;
  if (grid > static_cast<int64_t>(sm_count) * 16) grid = static_cast<int64_t>(sm_count) * 16;
  split_bf16x3_kernel<<<static_cast<int>(grid), 256, 0, stream>>>(src, n_rows, dim, ld_src, dst, ld_dst);
  return cudaGetLastError();
}

// ---- small fills ----------------------------------------------------------------------------
template <typename X>
__global__ void fill_kernel(X* p, X v, int64_t n) {
  const int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i < n) p[i] = v;
}
cudaError_t launch_fill_u32(uint32_t* p, uint32_t v, int64_t n, cudaStream_t stream) {
  if (n <= 0) return cudaSuccess;
  fill_kernel<uint32_t><<<static_cast<int>((n + 255) / 256), 256, 0, stream>>>(p, v, n);
  return cudaGetLastError();
}

// ---- row filter: bool mask -> allow-list bitmap ------------------------------------------------
// One warp per 32-row word: a ballot over the mask bytes is the word; words past the last row are
// written as 0 (the padding the scan kernels rely on).  *count (zeroed by the caller) += popcount.
__global__ void __launch_bounds__(256) pack_row_filter_kernel(const uint8_t* __restrict__ allowed, int64_t n_rows,
                                                              uint32_t* __restrict__ words, int64_t n_words,
                                                              unsigned long long* count) {
  const int lane = threadIdx.x & 31;
  const int64_t n_warps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
  uint32_t n = 0;
  for (int64_t w = (blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x) >> 5; w < n_words; w += n_warps) {
    const int64_t r = w * 32 + lane;
    const uint32_t b = __ballot_sync(0xffffffffu, r < n_rows && allowed[r] != 0);
    if (lane == 0) { words[w] = b; n += __popc(b); }
  }
  if (lane == 0 && n) atomicAdd(count, static_cast<unsigned long long>(n));
}
cudaError_t launch_pack_row_filter(const uint8_t* allowed, int64_t n_rows, uint32_t* words, int64_t n_words,
                                   unsigned long long* count, int sm_count, cudaStream_t stream) {
  if (n_words <= 0) return cudaSuccess;
  int64_t grid = (n_words * 32 + 255) / 256;
  if (grid > static_cast<int64_t>(sm_count) * 8) grid = static_cast<int64_t>(sm_count) * 8;
  pack_row_filter_kernel<<<static_cast<int>(grid), 256, 0, stream>>>(allowed, n_rows, words, n_words, count);
  return cudaGetLastError();
}

}  // namespace mmrs
