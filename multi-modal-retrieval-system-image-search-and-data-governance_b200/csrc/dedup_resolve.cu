// dedup_resolve.cu -- the greedy first-keeper decision of tool/find_repeated_in_same_folder.py:76-95 on
// the device (mmrs_resolve_duplicates in api.cu).
//
// The host walk visits the rows in `order`; a row with an already kept neighbour is a duplicate of the
// earliest kept one, any other row is kept.  In rank space (rank[order[t]] = t) that is: a rank is KEPT iff
// none of its lower-ranked neighbours is kept, and a removed rank's representative is its lowest-ranked
// kept neighbour (kept ranks are kept in rank order).  Both follow by induction on rank.
//   rank     rank[order[t]] = t by atomic exchange against a sentinel: a repeated id is seen
//   orient   pair (i, j) -> edge (max rank, min rank); self-pairs and pairs with a row outside `order` become
//            a sentinel edge that sorts past every rank (an unranked row is never kept and never blocks)
//   sort     mmrs_sort_pairs on the oriented edges: each rank's lower neighbours are contiguous, ascending
//   offsets  off[r] = first edge of rank r (a lower bound per rank), cursor[r] = off[r]
//   rounds   every undecided rank moves its cursor past REMOVED neighbours: a KEPT neighbour makes it
//            REMOVED with that neighbour as representative, an UNDECIDED one ends its turn, the end of its
//            list makes it KEPT.  The undecided ranks go to the next round's worklist.
//   tail     one warp sweeps the remaining ranks in ascending order (exact by the definition above)
//   map back representative[order[r]] = order[res[r]]
//
// res[r] is the decision of rank r: -1 undecided, r kept, else the representative's rank (< r).  A rank
// moves from undecided to its final value once, with one 32-bit store, so a round that reads a neighbour
// while another thread decides it sees one of the two values and is right either way: undecided only ends
// the turn early.  The lowest undecided rank has only decided lower neighbours, so every round decides at
// least one rank or moves a cursor.  No thread ever waits for another: kernel boundaries and the warp's own
// program order are the only ordering used.
#include "common.cuh"

namespace mmrs {

constexpr int kResolveThreads = 256;
constexpr int32_t kEdgeSentinel = 0x7fffffff;   // above every rank (n_order < 2^31)
// a round looks at most this many edges of one rank; the rest waits for the next round or the tail, which
// reads neighbour lists 32 edges at a time
constexpr int kRoundEdgeBudget = 32;

static int resolve_grid(int64_t n, int sm_count) {
  int64_t g = (n + kResolveThreads - 1) / kResolveThreads;
  const int64_t cap = static_cast<int64_t>(sm_count) * 8;
  if (g > cap) g = cap;
  return static_cast<int>(g < 1 ? 1 : g);
}

__global__ void __launch_bounds__(kResolveThreads) resolve_rank_kernel(const int64_t* __restrict__ order, int64_t n_order,
                                                                      int64_t n_items, uint32_t* __restrict__ rank,
                                                                      int32_t* __restrict__ status) {
  for (int64_t t = blockIdx.x * static_cast<int64_t>(kResolveThreads) + threadIdx.x; t < n_order;
       t += static_cast<int64_t>(gridDim.x) * kResolveThreads) {
    const int64_t v = order ? order[t] : t;
    if (v < 0 || v >= n_items) {
      atomicOr(status, kResolveOrderRange);
      continue;
    }
    if (atomicExch(rank + v, static_cast<uint32_t>(t)) != 0xffffffffu) atomicOr(status, kResolveOrderRepeat);
  }
}

__global__ void __launch_bounds__(kResolveThreads) resolve_orient_kernel(const int64_t* __restrict__ pairs, int64_t n_pairs,
                                                                        int64_t n_items, const uint32_t* __restrict__ rank,
                                                                        int64_t* __restrict__ edges,
                                                                        int32_t* __restrict__ status) {
  for (int64_t p = blockIdx.x * static_cast<int64_t>(kResolveThreads) + threadIdx.x; p < n_pairs;
       p += static_cast<int64_t>(gridDim.x) * kResolveThreads) {
    const int64_t i = pairs[2 * p], j = pairs[2 * p + 1];
    int64_t hi = kEdgeSentinel, lo = kEdgeSentinel;
    if (i < 0 || i >= n_items || j < 0 || j >= n_items) {
      atomicOr(status, kResolvePairRange);
    } else {
      const uint32_t ri = rank[i], rj = rank[j];
      if (ri != 0xffffffffu && rj != 0xffffffffu && ri != rj) {
        hi = ri > rj ? ri : rj;
        lo = ri > rj ? rj : ri;
      }
    }
    edges[2 * p] = hi;
    edges[2 * p + 1] = lo;
  }
}

// off[r] = first sorted edge whose high end is >= r, r in [0, n_order]; cursor[r] = off[r]
__global__ void __launch_bounds__(kResolveThreads) resolve_offsets_kernel(const int64_t* __restrict__ edges, int64_t n_edges,
                                                                         int64_t n_order, int64_t* __restrict__ off,
                                                                         int64_t* __restrict__ cursor) {
  for (int64_t r = blockIdx.x * static_cast<int64_t>(kResolveThreads) + threadIdx.x; r <= n_order;
       r += static_cast<int64_t>(gridDim.x) * kResolveThreads) {
    int64_t a = 0, b = n_edges;
    while (a < b) {
      const int64_t m = (a + b) >> 1;
      if (edges[2 * m] < r) a = m + 1; else b = m;
    }
    off[r] = a;
    if (r < n_order) cursor[r] = a;
  }
}

// One round over the worklist (wl_in == nullptr: every rank 0..n_first-1).  Undecided ranks are appended to
// wl_out in arrival order.
__global__ void __launch_bounds__(kResolveThreads) resolve_round_kernel(const int32_t* __restrict__ wl_in,
                                                                       const uint32_t* __restrict__ cnt_in, int64_t n_first,
                                                                       int32_t* __restrict__ wl_out, uint32_t* cnt_out,
                                                                       const int64_t* __restrict__ off,
                                                                       const int64_t* __restrict__ edges,
                                                                       int64_t* __restrict__ cursor, int32_t* res) {
  const int64_t n = wl_in ? static_cast<int64_t>(*cnt_in) : n_first;
  const int lane = threadIdx.x & 31;
  for (int64_t i = blockIdx.x * static_cast<int64_t>(kResolveThreads) + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * kResolveThreads) {
    const int32_t r = wl_in ? wl_in[i] : static_cast<int32_t>(i);
    int64_t c = cursor[r];
    const int64_t end = off[r + 1];
    int32_t out = -1;
    for (int budget = kRoundEdgeBudget; c < end && budget > 0; ++c, --budget) {
      const int32_t u = static_cast<int32_t>(edges[2 * c + 1]);
      const int32_t s = __ldcg(res + u);          // L2: the freshest value another SM may have written
      if (s < 0) break;                           // undecided: this rank's turn ends
      if (s == u) { out = u; break; }             // kept: the first kept neighbour in rank order
    }
    if (out < 0 && c == end) out = r;             // every lower neighbour removed (or none): kept
    if (out >= 0) {
      res[r] = out;
    } else {
      cursor[r] = c;
    }
    const bool append = out < 0;
    const unsigned act = __activemask();
    const unsigned m = __ballot_sync(act, append);
    const int leader = __ffs(act) - 1;
    uint32_t base = 0;
    if (lane == leader && m) base = atomicAdd(cnt_out, static_cast<uint32_t>(__popc(m)));
    base = __shfl_sync(act, base, leader);
    if (append) wl_out[base + __popc(m & ((1u << lane) - 1u))] = r;
  }
}

// range[0] = max(~r), range[1] = max(r + 1) over the worklist: the lowest rank is ~range[0], range[1] is one past
// the highest (both words start at 0)
__global__ void __launch_bounds__(kResolveThreads) resolve_worklist_range_kernel(const int32_t* __restrict__ wl,
                                                                                const uint32_t* __restrict__ cnt,
                                                                                uint32_t* __restrict__ range) {
  const int64_t n = *cnt;
  uint32_t lo = 0, hi = 0;
  for (int64_t i = blockIdx.x * static_cast<int64_t>(kResolveThreads) + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * kResolveThreads) {
    const uint32_t r = static_cast<uint32_t>(wl[i]);
    lo = max(lo, ~r);
    hi = max(hi, r + 1u);
  }
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) {
    lo = max(lo, __shfl_xor_sync(0xffffffffu, lo, o));
    hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, o));
  }
  if ((threadIdx.x & 31) == 0 && hi) {
    atomicMax(range, lo);
    atomicMax(range + 1, hi);
  }
}

__device__ __forceinline__ int32_t load_res(const int32_t* p) { return *reinterpret_cast<const volatile int32_t*>(p); }

// The tail: one warp decides every undecided rank of [lo, hi) in ascending order.  All lower ranks are decided
// when a rank's turn comes, so its first kept neighbour (or none) is final.  The decisions of the current
// 32-rank chunk stay in registers (lane j holds rank base + j) and are read by shuffle; older ones are in res.
__global__ void __launch_bounds__(32) resolve_tail_kernel(const uint32_t* __restrict__ range,
                                                          const int64_t* __restrict__ off,
                                                          const int64_t* __restrict__ edges,
                                                          const int64_t* __restrict__ cursor, int32_t* res) {
  const int lane = threadIdx.x;
  const int64_t lo = static_cast<int64_t>(~range[0]), hi = range[1];
  for (int64_t base = lo; base < hi; base += 32) {
    const int64_t r = base + lane;
    const bool inb = r < hi;
    int32_t mine = inb ? load_res(res + r) : 0;
    const unsigned todo = __ballot_sync(0xffffffffu, inb && mine < 0);
    if (!todo) continue;
    int64_t c = 0, e = 0;
    int32_t u0 = -1;
    if ((todo >> lane) & 1u) {
      c = cursor[r];
      e = off[r + 1];
      if (c < e) u0 = static_cast<int32_t>(edges[2 * c + 1]);
    }
    for (unsigned left = todo; left; left &= left - 1u) {
      const int j = __ffs(left) - 1;
      const int64_t cj = __shfl_sync(0xffffffffu, c, j), ej = __shfl_sync(0xffffffffu, e, j);
      int32_t found = -1;
      if (ej - cj == 1) {                       // one neighbour left: its first edge was loaded with the chunk
        const int32_t u = __shfl_sync(0xffffffffu, u0, j);
        const int32_t near = __shfl_sync(0xffffffffu, mine, (u - static_cast<int32_t>(base)) & 31);
        const int32_t s = u >= base ? near : load_res(res + u);
        if (s == u) found = u;
      } else {
        for (int64_t cc = cj; cc < ej; cc += 32) {
          const int64_t k = cc + lane;
          const int32_t u = k < ej ? static_cast<int32_t>(edges[2 * k + 1]) : -1;
          const int32_t near = __shfl_sync(0xffffffffu, mine, (u - static_cast<int32_t>(base)) & 31);
          const int32_t s = u < 0 ? -1 : (u >= base ? near : load_res(res + u));
          const unsigned kept = __ballot_sync(0xffffffffu, u >= 0 && s == u);
          if (kept) {
            found = __shfl_sync(0xffffffffu, u, __ffs(kept) - 1);   // lowest edge = lowest rank
            break;
          }
        }
      }
      if (lane == j) mine = found >= 0 ? found : static_cast<int32_t>(base + j);
      __syncwarp();
    }
    if ((todo >> lane) & 1u) res[r] = mine;
    __syncwarp();
  }
}

__global__ void __launch_bounds__(kResolveThreads) resolve_map_back_kernel(const int64_t* __restrict__ order, int64_t n_order,
                                                                          int64_t n_items, const int32_t* __restrict__ res,
                                                                          int64_t* __restrict__ rep) {
  for (int64_t r = blockIdx.x * static_cast<int64_t>(kResolveThreads) + threadIdx.x; r < n_order;
       r += static_cast<int64_t>(gridDim.x) * kResolveThreads) {
    const int64_t v = order ? order[r] : r;
    const int32_t s = res[r];
    if (v < 0 || v >= n_items || s < 0) continue;   // only after an error the status word reports
    rep[v] = order ? order[s] : s;
  }
}

cudaError_t launch_resolve_rank(const int64_t* order, int64_t n_order, int64_t n_items, uint32_t* rank, int32_t* status,
                                int sm_count, cudaStream_t stream) {
  if (n_order < 1) return cudaSuccess;
  resolve_rank_kernel<<<resolve_grid(n_order, sm_count), kResolveThreads, 0, stream>>>(order, n_order, n_items, rank,
                                                                                          status);
  return cudaGetLastError();
}

cudaError_t launch_resolve_orient(const int64_t* pairs, int64_t n_pairs, int64_t n_items, const uint32_t* rank,
                                  int64_t* edges, int32_t* status, int sm_count, cudaStream_t stream) {
  if (n_pairs < 1) return cudaSuccess;
  resolve_orient_kernel<<<resolve_grid(n_pairs, sm_count), kResolveThreads, 0, stream>>>(pairs, n_pairs, n_items, rank,
                                                                                            edges, status);
  return cudaGetLastError();
}

cudaError_t launch_resolve_offsets(const int64_t* edges, int64_t n_edges, int64_t n_order, int64_t* off, int64_t* cursor,
                                   int sm_count, cudaStream_t stream) {
  resolve_offsets_kernel<<<resolve_grid(n_order + 1, sm_count), kResolveThreads, 0, stream>>>(edges, n_edges, n_order,
                                                                                                 off, cursor);
  return cudaGetLastError();
}

cudaError_t launch_resolve_round(const int32_t* wl_in, const uint32_t* cnt_in, int64_t n_first, int64_t n_bound,
                                 int32_t* wl_out, uint32_t* cnt_out, const int64_t* off, const int64_t* edges,
                                 int64_t* cursor, int32_t* res, int sm_count, cudaStream_t stream) {
  cudaError_t e = cudaMemsetAsync(cnt_out, 0, sizeof(uint32_t), stream);
  if (e != cudaSuccess || n_bound < 1) return e;
  resolve_round_kernel<<<resolve_grid(n_bound, sm_count), kResolveThreads, 0, stream>>>(wl_in, cnt_in, n_first, wl_out,
                                                                                           cnt_out, off, edges, cursor,
                                                                                           res);
  return cudaGetLastError();
}

cudaError_t launch_resolve_tail(const int32_t* wl, const uint32_t* cnt, int64_t n_bound, uint32_t* range,
                                const int64_t* off, const int64_t* edges, const int64_t* cursor, int32_t* res,
                                int sm_count, cudaStream_t stream) {
  cudaError_t e = cudaMemsetAsync(range, 0, 2 * sizeof(uint32_t), stream);
  if (e != cudaSuccess || n_bound < 1) return e;
  resolve_worklist_range_kernel<<<resolve_grid(n_bound, sm_count), kResolveThreads, 0, stream>>>(wl, cnt, range);
  resolve_tail_kernel<<<1, 32, 0, stream>>>(range, off, edges, cursor, res);
  return cudaGetLastError();
}

cudaError_t launch_resolve_map_back(const int64_t* order, int64_t n_order, int64_t n_items, const int32_t* res,
                                    int64_t* rep, int sm_count, cudaStream_t stream) {
  if (n_order < 1) return cudaSuccess;
  resolve_map_back_kernel<<<resolve_grid(n_order, sm_count), kResolveThreads, 0, stream>>>(order, n_order, n_items, res,
                                                                                              rep);
  return cudaGetLastError();
}

}  // namespace mmrs
