// host.h -- host-side plumbing of the extern "C" entry points, shared by every .cu file that defines some:
// the error state, launch counting and profiling, the device query, the pinned status word, argument
// checks and the workspace carver.  The library-wide state is C++17 inline variables, so every file sees
// the same error text, launch counter and profile records.
#pragma once
#include <stdarg.h>
#include <stdio.h>

#include <atomic>
#include <mutex>
#include <vector>

#include "common.cuh"

namespace mmrs {

inline thread_local char g_err[512] = "";

inline int fail(int code, const char* fmt, ...) {
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
inline std::atomic<long long> g_launches{0};
struct ProfRec { cudaEvent_t e0, e1; int32_t kind; int64_t bytes; int64_t flops; };
inline std::mutex g_prof_mu;
inline std::vector<ProfRec> g_prof;
inline std::atomic<int> g_prof_on{0};

#define MMRS_LAUNCH(expr)        \
  do {                           \
    g_launches.fetch_add(1);     \
    MMRS_CUDA(expr);             \
  } while (0)

template <typename F>
int profiled_launch(int32_t kind, int64_t bytes, int64_t flops, cudaStream_t stream, F launch) {
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

struct DeviceInfo {
  int device = -1;
  int sm_count = 0;
  int cc_major = 0;
};

inline int current_device(DeviceInfo* info) {
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

// 32 bytes of pinned host memory per thread that the synchronous entry points read status words and
// counts back into; nullptr when the allocation failed
inline int32_t* pinned_status() {
  static thread_local int32_t* h = nullptr;
  if (!h) {
    if (cudaHostAlloc(reinterpret_cast<void**>(&h), 8 * sizeof(int32_t), cudaHostAllocDefault) != cudaSuccess)
      h = nullptr;
  }
  return h;
}

inline int check_matrix(const void* p, int64_t n_rows, int32_t dim, int64_t ld, int32_t dtype, const char* what) {
  if (!p) return fail(MMRS_ERR_ARG, "%s pointer is null", what);
  if (n_rows < 1) return fail(MMRS_ERR_ARG, "%s has %lld rows", what, (long long)n_rows);
  if (n_rows > 0xffffffffll) return fail(MMRS_ERR_ARG, "%s: more than 2^32 rows per shard", what);
  if (dtype != MMRS_DTYPE_F32 && dtype != MMRS_DTYPE_BF16 && dtype != MMRS_DTYPE_BF16X3 && dtype != MMRS_DTYPE_I8)
    return fail(MMRS_ERR_ARG, "%s dtype %d unknown", what, dtype);
  if (dtype == MMRS_DTYPE_I8) {   // codes [dim], the row's scale at byte dim (include/mmrs_b200.h, "int8 galleries")
    if (dim < 1 || dim % 16 != 0)
      return fail(MMRS_ERR_ARG, "%s: int8 dim %d must be a positive multiple of 16 (zero codes pad it)", what, dim);
    if (ld < dim + 16 || ld % 16 != 0)
      return fail(MMRS_ERR_ARG, "%s: int8 row stride %lld must be >= dim + 16 and a multiple of 16 bytes", what,
                  (long long)ld);
    if (reinterpret_cast<uintptr_t>(p) % 16 != 0)
      return fail(MMRS_ERR_ARG, "%s pointer must be 16-byte aligned", what);
    return MMRS_OK;
  }
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

// ---- caller-owned workspaces ---------------------------------------------------------------------
inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Bump allocator over a workspace: every piece starts on a 256-byte boundary.  With a null base it
// hands out null pointers and only sums the sizes, so a *_workspace_bytes query and the entry point
// that carves the buffer run the same code and cannot disagree on the layout.
struct Carver {
  char* base;
  size_t off = 0;
  explicit Carver(void* b) : base(static_cast<char*>(b)) {}
  template <typename T>
  T* take(size_t bytes) {
    char* p = base ? base + off : nullptr;
    off += align_up(bytes, 256);
    return reinterpret_cast<T*>(p);
  }
};

// At least `need` bytes; 256-byte alignment where the entry point's layout assumes it.
inline int check_workspace(const void* ws, size_t bytes, size_t need, bool aligned = true) {
  if (!ws || bytes < need) return fail(MMRS_ERR_WORKSPACE, "workspace %zu bytes, need %zu", bytes, need);
  if (aligned && reinterpret_cast<uintptr_t>(ws) % 256 != 0)
    return fail(MMRS_ERR_WORKSPACE, "workspace must be 256-byte aligned");
  return MMRS_OK;
}

}  // namespace mmrs
