// select.cu -- K3/K4: exact per-query top-k over a list of unique u64 keys.
//
// One 1024-thread CTA per query.  The list (survivors of the previous phase + the keys the scan
// appended, or a dense seed sample) is read once, coalesced, into registers.  The k-th largest
// key is then found by a bit-wise descent, two bits per step: the block counts how many keys are
// >= each of three pivots (register compares + one REDUX per warp + one barrier) and keeps the
// largest pivot that still has >= k keys above it; leading bits shared by all keys are skipped
// and the walk stops as soon as a pivot has exactly k keys above it.  No shared-memory atomics:
// a histogram radix select costs one ATOMS per key, which at ~50 clk per warp-wide ATOMS made the
// first version of this kernel 11-20 us per call (profiles/r01_launches_b16.csv).
// The k winners are ranked by counting (rank = #keys greater), which sorts them without any
// barrier-separated network stages, and are written either back to the front of the list with
// the new score bound (between scan phases) or as (values, indices) in torch.topk order
// (code/utils.py:17: largest, sorted).  Keys are (score, ~row), so the result is exactly "score
// descending, row ascending" whatever order the scan kernels appended the candidates in.
//
// The same kernel merges the per-GPU lists after the all-gather (mmrs_topk_merge): pack_keys
// turns (value, global index) pairs back into keys.
#include "common.cuh"

namespace mmrs {

constexpr int kSelThreads = 1024;
constexpr int kSelWarps = kSelThreads / 32;
constexpr int kSelMaxK = 1024;
constexpr int kSelMaxKpt = 16;                     // register-resident lists: up to 16 Ki keys
constexpr int kSelWinners = kSelMaxK + kSelMaxK / 4 + 8;
constexpr int kSelBucket = 512;                    // bucket small enough for one warp to finish

struct SelShared {
  uint32_t warp_cnt[2][kSelWarps];   // packed per-warp pivot counts, double buffered
  uint32_t wide_cnt[3][kSelWarps];   // generic path: unpacked
  uint64_t red_min[kSelWarps];
  uint64_t red_max[kSelWarps];
  uint32_t n_out;
  uint32_t n_bucket;
  uint64_t thr_key;
  uint64_t bucket[kSelBucket];
  uint64_t winners[kSelWinners];
};

// Between phases only a BOUND is needed: any pivot with at least k and at most this many keys
// above it ends the descent; the (unsorted) keys above it become the next list.
__device__ __forceinline__ uint32_t relaxed_limit(uint32_t k) { return k + k / 4 + 8; }

// The walk towards the k-th largest key.  State: `prefix` with `pos` undecided low bits;
// ge = #keys >= prefix (>= k), above = #keys >= prefix + 2^pos (< k).  One step tries the three
// pivots prefix | d << (pos-2), d = 1..3, and keeps the largest with >= k keys at or above it.
struct Walk {
  uint64_t prefix;
  int pos;
  uint32_t ge, above;
};
__device__ __forceinline__ void walk_step(Walk& w, uint32_t k, uint32_t t1, uint32_t t2, uint32_t t3, int bits) {
  const int shift = w.pos - bits;
  // counts at the four digit boundaries, descending digit: t[3], t[2], t[1], ge
  if (bits == 2 && t3 >= k) { w.prefix |= 3ull << shift; w.ge = t3; /* above unchanged */ }
  else if (bits == 2 && t2 >= k) { w.prefix |= 2ull << shift; w.ge = t2; w.above = t3; }
  else if (t1 >= k) { w.prefix |= 1ull << shift; w.ge = t1; w.above = bits == 2 ? t2 : w.above; }
  else { w.above = t1; }
  w.pos = shift;
}

template <int KPT>
__device__ __forceinline__ void select_body(const SelectParams& p, SelShared& sh, uint64_t* list, uint32_t n,
                                            int q) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t k = p.k;
  const uint32_t limit = p.final_pass ? k : relaxed_limit(k);
  constexpr bool in_regs = KPT > 0;
  constexpr int R = in_regs ? KPT : 1;

  const int32_t seg_len = p.seg_len;
  const uint64_t* seg_base = p.cand + static_cast<int64_t>(q) * seg_len;
  auto load = [&](uint32_t idx) -> uint64_t {
    if (seg_len == 0) return list[idx];
    return seg_base[static_cast<int64_t>(idx / seg_len) * p.seg_stride + idx % seg_len];
  };
  uint64_t key[R];
  if constexpr (in_regs) {
#pragma unroll
    for (int i = 0; i < KPT; ++i) {
      const uint32_t idx = tid + i * kSelThreads;
      key[i] = idx < n ? load(idx) : 0ull;   // 0 is below every real key
    }
  }
  auto for_each_key = [&](auto&& f) {
    if constexpr (in_regs) {
#pragma unroll
      for (int i = 0; i < KPT; ++i) f(key[i]);
    } else {
      // block-uniform trip count (the callbacks use warp collectives); 0 pads the tail
      for (uint32_t base = 0; base < n; base += kSelThreads) {
        const uint32_t idx = base + tid;
        f(idx < n ? load(idx) : 0ull);
      }
    }
  };

  // ---- leading bits shared by every key (zeros = padding / rows past the gallery end are ignored) --
  uint64_t mn = ~0ull, mx = 0ull;
  for_each_key([&](uint64_t x) {
    if (x != 0ull) { mn = x < mn ? x : mn; mx = x > mx ? x : mx; }
  });
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) {
    const uint64_t a = __shfl_xor_sync(0xffffffffu, mn, o);
    const uint64_t b = __shfl_xor_sync(0xffffffffu, mx, o);
    mn = a < mn ? a : mn;
    mx = b > mx ? b : mx;
  }
  if (lane == 0) { sh.red_min[warp] = mn; sh.red_max[warp] = mx; }
  if (tid == 0) { sh.n_out = 0; sh.n_bucket = 0; }
  __syncthreads();
  mn = sh.red_min[lane];
  mx = sh.red_max[lane];
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) {
    const uint64_t a = __shfl_xor_sync(0xffffffffu, mn, o);
    const uint64_t b = __shfl_xor_sync(0xffffffffu, mx, o);
    mn = a < mn ? a : mn;
    mx = b > mx ? b : mx;
  }

  uint64_t thr_key;
  if (n <= limit) {
    thr_key = mn;                        // every real key is selected
  } else {
    const uint64_t diff = mn ^ mx;
    Walk w;
    w.pos = diff == 0 ? 0 : 64 - __clzll(static_cast<long long>(diff));   // undecided low bits
    w.prefix = w.pos >= 64 ? 0ull : (mx >> w.pos) << w.pos;
    w.ge = n;       // zeros included: harmless, they are never >= a pivot
    w.above = 0;
    int buf = 0;
    // ---- phase A: block-wide steps until the bucket [prefix, prefix + 2^pos) is small ------------
    while (w.pos > 0 && w.ge > limit && (w.ge - w.above) > kSelBucket) {
      const int bits = w.pos >= 2 ? 2 : 1;
      const int shift = w.pos - bits;
      const uint64_t p1 = w.prefix | (1ull << shift);
      const uint64_t p2 = w.prefix | (2ull << shift);     // only meaningful when bits == 2
      const uint64_t p3 = w.prefix | (3ull << shift);
      uint32_t c1 = 0, c2 = 0, c3 = 0;
      for_each_key([&](uint64_t x) {
        c1 += x >= p1;
        c2 += x >= p2;
        c3 += x >= p3;
      });
      uint32_t t1, t2, t3;
      if constexpr (in_regs) {
        // per-warp sums are <= 32 * 16 = 512: three 10-bit fields in one REDUX
        const uint32_t packed = __reduce_add_sync(0xffffffffu, c1 | (c2 << 10) | (c3 << 20));
        if (lane == 0) sh.warp_cnt[buf][warp] = packed;
        __syncthreads();
        const uint32_t v = sh.warp_cnt[buf][lane];
        t1 = __reduce_add_sync(0xffffffffu, v & 1023u);
        t2 = __reduce_add_sync(0xffffffffu, (v >> 10) & 1023u);
        t3 = __reduce_add_sync(0xffffffffu, v >> 20);
        buf ^= 1;
      } else {
        c1 = __reduce_add_sync(0xffffffffu, c1);
        c2 = __reduce_add_sync(0xffffffffu, c2);
        c3 = __reduce_add_sync(0xffffffffu, c3);
        __syncthreads();                       // previous step's readers are done
        if (lane == 0) { sh.wide_cnt[0][warp] = c1; sh.wide_cnt[1][warp] = c2; sh.wide_cnt[2][warp] = c3; }
        __syncthreads();
        t1 = __reduce_add_sync(0xffffffffu, sh.wide_cnt[0][lane]);
        t2 = __reduce_add_sync(0xffffffffu, sh.wide_cnt[1][lane]);
        t3 = __reduce_add_sync(0xffffffffu, sh.wide_cnt[2][lane]);
      }
      walk_step(w, k, t1, t2, t3, bits);
    }
    // ---- phase B: one warp finishes on the bucket's keys ------------------------------------------
    if (w.pos > 0 && w.ge > limit) {
      const uint64_t lo = w.prefix;
      const uint64_t hi_excl_minus1 = w.prefix | ((w.pos >= 64 ? ~0ull : ((1ull << w.pos) - 1ull)));
      for_each_key([&](uint64_t x) {
        const bool in = x >= lo && x <= hi_excl_minus1 && x != 0ull;
        const uint32_t m = __ballot_sync(0xffffffffu, in);
        if (m) {
          uint32_t base = 0;
          if (lane == 0) base = atomicAdd(&sh.n_bucket, static_cast<uint32_t>(__popc(m)));
          base = __shfl_sync(0xffffffffu, base, 0);
          if (in) sh.bucket[base + __popc(m & ((1u << lane) - 1u))] = x;   // count <= kSelBucket by construction
        }
      });
      __syncthreads();
      if (warp == 0) {
        const uint32_t nb = sh.n_bucket;
        for (uint32_t idx = nb + lane; idx < kSelBucket; idx += 32) sh.bucket[idx] = 0ull;   // pad
        __syncwarp();
        const uint32_t n_it = (nb + 31) / 32;    // warp-uniform
        const uint32_t base_above = w.above;     // keys above the bucket count for every pivot
        while (w.pos > 0 && w.ge > limit) {
          const int bits = w.pos >= 2 ? 2 : 1;
          const int shift = w.pos - bits;
          const uint64_t p1 = w.prefix | (1ull << shift);
          const uint64_t p2 = w.prefix | (2ull << shift);
          const uint64_t p3 = w.prefix | (3ull << shift);
          uint32_t c1 = 0, c2 = 0, c3 = 0;
          for (uint32_t i = 0; i < n_it; ++i) {       // keys stay in shared memory: no register cost
            const uint64_t x = sh.bucket[lane + i * 32];
            c1 += x >= p1;
            c2 += x >= p2;
            c3 += x >= p3;
          }
          const uint32_t packed = __reduce_add_sync(0xffffffffu, c1 | (c2 << 10) | (c3 << 20));
          walk_step(w, k, base_above + (packed & 1023u), base_above + ((packed >> 10) & 1023u),
                    base_above + (packed >> 20), bits);
        }
        if (lane == 0) sh.thr_key = w.prefix;
      }
      __syncthreads();
      thr_key = sh.thr_key;
    } else {
      thr_key = w.prefix;
    }
  }

  // ---- gather the winners -------------------------------------------------------------------------
  __syncthreads();
  for_each_key([&](uint64_t x) {
    const bool win = x >= thr_key && x != 0ull;
    const uint32_t m = __ballot_sync(0xffffffffu, win);
    if (m) {
      uint32_t base = 0;
      if (lane == 0) base = atomicAdd(&sh.n_out, static_cast<uint32_t>(__popc(m)));
      base = __shfl_sync(0xffffffffu, base, 0);
      if (win) {
        const uint32_t slot = base + __popc(m & ((1u << lane) - 1u));
        if (slot < kSelWinners) sh.winners[slot] = x;
      }
    }
  });
  __syncthreads();
  const uint32_t n_win = sh.n_out;
  if ((n_win < k && !p.pad_short) || n_win > limit) {  // uniqueness violated (bug guard)
    if (tid == 0) atomicOr(p.flags, kFlagShort);
    if (n_win > limit) return;
  }
  const bool short_list = p.pad_short && n_win < k;   // fewer than k allowed rows so far

  if (p.final_pass) {
    // rank by counting: position = number of winners with a larger key
    for (uint32_t i = tid; i < n_win; i += kSelThreads) {
      const uint64_t mine = sh.winners[i];
      uint32_t rank = 0;
      for (uint32_t j = 0; j < n_win; ++j) rank += sh.winners[j] > mine;
      const int64_t grow = static_cast<int64_t>(key_row(mine)) + p.index_offset;
      if (p.out_values) p.out_values[static_cast<int64_t>(q) * k + rank] = key_score(mine);
      if (p.out_indices) p.out_indices[static_cast<int64_t>(q) * k + rank] = grow;
      const uint64_t gkey = (mine & 0xffffffff00000000ull) | static_cast<uint64_t>(~static_cast<uint32_t>(grow));
      if (p.out_keys) p.out_keys[static_cast<int64_t>(q) * k + rank] = gkey;
      if (p.g_role == 1) {
        // fused all-gather: store the key straight into every rank's gather buffer over NVLink
        const int64_t off = static_cast<int64_t>(p.g_rank) * p.g_list_stride + static_cast<int64_t>(q) * k + rank;
        for (int r = 0; r < p.g_world; ++r) p.g_peer_bufs[r][off] = gkey;
      }
    }
    if (short_list) {
      // every position still gets written (a shard's list keeps exactly k entries; key 0 merges as nothing)
      for (uint32_t i = n_win + tid; i < k; i += kSelThreads) {
        const int64_t o = static_cast<int64_t>(q) * k + i;
        if (p.out_values) p.out_values[o] = __int_as_float(0xff800000);
        if (p.out_indices) p.out_indices[o] = -1;
        if (p.out_keys) p.out_keys[o] = 0ull;
        if (p.g_role == 1) {
          const int64_t off = static_cast<int64_t>(p.g_rank) * p.g_list_stride + o;
          for (int r = 0; r < p.g_world; ++r) p.g_peer_bufs[r][off] = 0ull;
        }
      }
    }
  } else {
    // next list = the winners (unsorted); bound = score part of the pivot (<= every winner's score).
    // Fewer than k winners: no bound yet, the next phase appends every (allowed) row.
    for (uint32_t i = tid; i < n_win; i += kSelThreads) list[i] = sh.winners[i];
    if (tid == 0) {
      p.cnt[q] = n_win;
      p.thr[q] = short_list ? __int_as_float(0xff800000) : key_score(thr_key);
    }
  }
}

__device__ void select_dispatch(const SelectParams& p, SelShared& sh, uint64_t* list, int q);

// The waits of the fused all-gather run in kernels of ONE warp, never inside the Q-CTA select
// kernels: a select grid that spins occupies every SM once Q >= the SM count, and two searches in
// flight on two streams could then wait for each other across ranks (rank A's slot-1 merge holds
// A's SMs waiting for B's slot-1 keys while B's slot-2 merge holds B's SMs waiting for A's slot-2
// keys, whose scan cannot get an SM).  A one-warp waiter leaves the machine to the scans.
//   gather_wait_kernel  consumer side: every rank's keys of this epoch have landed here (ready >= epoch)
//   (the producer side -- every rank has merged the previous use of this slot, ack >= epoch - 1 --
//    is waited for by block 0 of prep_queries_kernel, the first kernel of the call)
__global__ void __launch_bounds__(32) gather_wait_kernel(const uint32_t* my_flags, int32_t world,
                                                         const uint32_t* epoch, int32_t* status, uint64_t timeout_ns) {
  pdl_wait();   // NOT launch_dependents: the merge select must not be resident while this spins
  if (threadIdx.x == 0) wait_all_ge(my_flags, world, *epoch, status, timeout_ns);
}

cudaError_t launch_gather_wait(const uint32_t* my_flags, int32_t world, const uint32_t* epoch, int32_t* status,
                               uint64_t timeout_ns, cudaStream_t stream) {
  return launch_pdl(gather_wait_kernel, dim3(1), dim3(32), 0, stream, my_flags, world, epoch, status, timeout_ns);
}

__global__ void __launch_bounds__(kSelThreads, 1) select_topk_kernel(const SelectParams p) {
  __shared__ SelShared sh;
  const int q = blockIdx.x;
  const int tid = threadIdx.x;
  uint64_t* list = p.cand + static_cast<int64_t>(q) * p.cap;
  pdl_launch_dependents();
  pdl_wait();   // the list and its length come from the preceding scan

  select_dispatch(p, sh, list, q);
  if (p.g_role != 0) {
    // Last CTA out publishes: status word + "ready" (producer) or "ack" (consumer) to every rank.
    // Ordering: every thread's peer stores precede the CTA barrier; thread 0's system-scope fence after the
    // barrier is cumulative over them (the pattern of a cooperative-groups grid sync), so ONE fence per CTA
    // orders the CTA's stores before its ticket -- not one per thread; the last CTA fences once more after its
    // ticket (it has observed every other CTA's) and then raises the flags with plain system-scope stores:
    // eight st.release.sys in a row would each wait for all earlier writes again (the final selects of an
    // 8-GPU search took 35-38 us against 11-13 us for the same select without the gather).
    __syncthreads();
    if (tid == 0) {
      __threadfence_system();
      const uint32_t done = atomicAdd(p.g_counter, 1u);
      if (done == gridDim.x - 1) {
        __threadfence_system();
        *p.g_counter = 0;
        const uint32_t epoch = *p.g_epoch;
        if (p.g_role == 1) {
          const uint64_t status = static_cast<uint64_t>(static_cast<uint32_t>(*reinterpret_cast<volatile int32_t*>(p.flags)));
          for (int r = 0; r < p.g_world; ++r)
            p.g_peer_bufs[r][static_cast<int64_t>(p.g_rank) * p.g_list_stride + p.g_status_index] = status;
        } else {
          // the ranks' status words are copied out of the peer-writable buffer BEFORE the ack lets
          // epoch + 1 producers overwrite it: the host reads this private snapshot
          const uint64_t* mine = p.g_peer_bufs[p.g_rank];
          for (int r = 0; r < p.g_world; ++r)
            p.g_status_out[r] = static_cast<uint32_t>(
                *reinterpret_cast<const volatile uint64_t*>(mine + static_cast<int64_t>(r) * p.g_list_stride + p.g_status_index));
        }
        __threadfence_system();   // status words / snapshot reads are ordered before the flags
        const int slot = (p.g_role == 1 ? 0 : p.g_world) + p.g_rank;
        for (int r = 0; r < p.g_world; ++r) st_relaxed_sys(p.g_peer_flags[r] + slot, epoch);
      }
    }
  }
}

__device__ __forceinline__ void select_dispatch_impl(const SelectParams& p, SelShared& sh, uint64_t* list, int q) {
  const int tid = threadIdx.x;
  uint32_t n;
  if (p.fixed_n >= 0) {
    n = static_cast<uint32_t>(p.fixed_n);
  } else {
    n = p.cnt[q];
    if (n > static_cast<uint32_t>(p.cap)) {
      if (tid == 0) atomicOr(p.flags, kFlagOverflow);
      n = p.cap;
    }
  }
  if (n < static_cast<uint32_t>(p.k) && !p.pad_short) {  // cannot happen on a correct unfiltered schedule
    if (tid == 0) atomicOr(p.flags, kFlagShort);
    return;
  }
  // Lists up to 16 Ki keys live in registers, KPT slots per thread (instantiated per size so that
  // a 2 000-key list does not pay for 16 predicated slots); longer ones (the exhaustive fallback)
  // are re-read from global memory at every step.
  const uint32_t kpt = (n + kSelThreads - 1) / kSelThreads;
  if (kpt <= 1) select_body<1>(p, sh, list, n, q);
  else if (kpt <= 2) select_body<2>(p, sh, list, n, q);
  else if (kpt <= 4) select_body<4>(p, sh, list, n, q);
  else if (kpt <= 8) select_body<8>(p, sh, list, n, q);
  else if (kpt <= kSelMaxKpt) select_body<16>(p, sh, list, n, q);
  else select_body<0>(p, sh, list, n, q);
}
__device__ void select_dispatch(const SelectParams& p, SelShared& sh, uint64_t* list, int q) {
  select_dispatch_impl(p, sh, list, q);
}

const void* select_kernel_handle() { return reinterpret_cast<const void*>(select_topk_kernel); }

cudaError_t launch_select(const SelectParams& p, int32_t n_queries, cudaStream_t stream) {
  if (n_queries <= 0) return cudaSuccess;
  if (p.k < 1 || p.k > kSelMaxK) return cudaErrorInvalidValue;
  return launch_pdl(select_topk_kernel, dim3(n_queries), dim3(kSelThreads), 0, stream, p);
}

// (value, global index) -> key lists laid out [n_queries, cap] with cap = n_lists * k_in.
__global__ void pack_keys_kernel(const float* __restrict__ values,
                                 const int64_t* __restrict__ indices, int32_t n_lists,
                                 int32_t n_queries, int32_t k_in, uint64_t* __restrict__ cand,
                                 int32_t cap) {
  const int64_t total = static_cast<int64_t>(n_lists) * n_queries * k_in;
  const int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i >= total) return;
  const int j = static_cast<int>(i % k_in);
  const int q = static_cast<int>((i / k_in) % n_queries);
  const int l = static_cast<int>(i / (static_cast<int64_t>(k_in) * n_queries));
  cand[static_cast<int64_t>(q) * cap + l * k_in + j] =
      make_key(values[i], static_cast<uint32_t>(indices[i]));
}

cudaError_t launch_pack_keys(const float* values, const int64_t* indices, int32_t n_lists,
                             int32_t n_queries, int32_t k_in, uint64_t* cand, int32_t cap,
                             cudaStream_t stream) {
  const int64_t total = static_cast<int64_t>(n_lists) * n_queries * k_in;
  if (total <= 0) return cudaSuccess;
  pack_keys_kernel<<<static_cast<int>((total + 255) / 256), 256, 0, stream>>>(
      values, indices, n_lists, n_queries, k_in, cand, cap);
  return cudaGetLastError();
}

}  // namespace mmrs
