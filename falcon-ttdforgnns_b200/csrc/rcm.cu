// rcm.cu -- reverse Cuthill-McKee order of a CSR graph on the device (SURVEY 8f-3), element for
// element the permutation of scipy.sparse.csgraph.reverse_cuthill_mckee(adj, symmetric_mode=False)
// that DGL's 'rcmk' reorder returns (adj = the CSR of in-neighbour lists).  scipy walks the graph
// node by node; the same order restated level-synchronously (oracle/rcm_oracle.py):
//
//   1. symmetrise   scipy forms adj + adj^T.  Canonical input (every in-list strictly increasing):
//                   row i = the distinct neighbours of i, ascending.  Any other input: row i = the
//                   distinct entries of [in-list of i as stored] ++ [every v with i in in-list(v),
//                   increasing v], in REVERSE order of first appearance.
//   2. degree       row length, + 1 for a self loop (int32).
//   3. seed ranks   numpy.argsort of the degrees, on the host by the caller (the tie order is
//                   numpy's and is not restated here).
//   4. components   the seed of a component is its node of smallest rank; components in increasing
//                   seed rank.
//   5. levels       level 0 = the seed; every unvisited neighbour j of level L = f[0..m) is owned by
//                   the smallest (p, k): p = position of the parent in f, k = position of j in the
//                   parent's row.  Level L + 1 = the owned nodes sorted by (p, degree(j), k).
//   6. order        components' levels concatenated in seed-rank order, then reversed.
//
// Here: (1) sort of (row, col) pairs with their appearance rank + unique-by-key + a per-row sort by
// appearance; (4) min-rank hooking with pointer jumping, whose converged label IS the seed rank;
// (5) every component at once, one level per step: 64-bit atomicMin election of (p << 32 | k), an
// order-preserving compaction of the winners (already in (p, k) order), a stable radix sort by
// (p, degree); (6) a stable sort of the level order by seed rank, reversed.  Everything runs on the
// caller's stream in the caller's workspace; the host reads back a handful of counts (the
// symmetrised size, one frontier size per BFS level, one flag per component round).
//
// Out of contract: a pair of nodes joined by 128 or more parallel edges (scipy sums int8 values;
// the sum can wrap to 0 and scipy then drops the entry), and an in-list of 2^31 or more entries.
#include <chrono>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_select.cuh>

#include "graph.cuh"

namespace ttg {
namespace {

constexpr uint32_t kFromTranspose = 0x80000000u;   // appearance rank of an adj^T entry: after the in-list

// ---- symmetrise ------------------------------------------------------------------------------------
// one warp per row v of the in-lists: (v, u) with its position in the list and (u, v) ranked after every
// in-list entry in increasing v.  A stable sort by (row, col) then keeps each pair's first appearance first.
__global__ void __launch_bounds__(256)
sym_emit_kernel(int64_t n, int64_t nnz, int colbits, const int64_t* __restrict__ indptr,
                const int32_t* __restrict__ indices, uint64_t* __restrict__ keys, uint32_t* __restrict__ vals,
                int32_t* __restrict__ flags) {
  const int64_t v = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (v >= n) return;
  int64_t lo, hi;
  if (!csr_row(indptr, n, nnz, v, &lo, &hi)) {
    flags[1] = 1;
    return;
  }
  for (int64_t e = lo + lane; e < hi; e += 32) {
    const int32_t u = __ldg(indices + e);
    if (u < 0 || u >= n) {
      flags[1] = 1;   // id out of range
      continue;
    }
    keys[e] = ((uint64_t)v << colbits) | (uint64_t)u;
    vals[e] = (uint32_t)(e - lo);
    keys[nnz + e] = ((uint64_t)u << colbits) | (uint64_t)v;
    vals[nnz + e] = kFromTranspose | (uint32_t)v;
    if (e + 1 < hi && __ldg(indices + e + 1) <= u) flags[0] = 1;   // not canonical
  }
}

// row r of the distinct (row, col) keys, sorted: its bounds by binary search; degree = length + self loop
__global__ void __launch_bounds__(256)
sym_rows_kernel(int64_t n, int64_t m, int colbits, const uint64_t* __restrict__ ukeys,
                int64_t* __restrict__ sym_indptr, int32_t* __restrict__ degree) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r > n) return;
  if (r == n) {
    sym_indptr[n] = m;
    return;
  }
  const int64_t lo = lower_bound_u64(ukeys, m, (uint64_t)r << colbits);
  const int64_t hi = lower_bound_u64(ukeys + lo, m - lo, (uint64_t)(r + 1) << colbits) + lo;
  const uint64_t self = ((uint64_t)r << colbits) | (uint64_t)r;
  const int64_t s = lower_bound_u64(ukeys + lo, hi - lo, self) + lo;
  sym_indptr[r] = lo;
  degree[r] = (int32_t)(hi - lo) + (s < hi && ukeys[s] == self ? 1 : 0);
}

// general input: key (row, reverse appearance) for the per-row sort, value the column
__global__ void __launch_bounds__(256)
sym_reverse_key_kernel(int64_t m, int colbits, const uint64_t* __restrict__ ukeys,
                       const uint32_t* __restrict__ uvals, uint64_t* __restrict__ keys,
                       uint32_t* __restrict__ cols) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= m) return;
  const uint64_t k = ukeys[i];
  keys[i] = ((k >> colbits) << 32) | (uint64_t)(0xFFFFFFFFu - uvals[i]);
  cols[i] = (uint32_t)(k & ((1ull << colbits) - 1));
}

// ---- components --------------------------------------------------------------------------------------
// label[v] = rank of v; node_of[r] = node of rank r; owner[v] = none; visited[v] = 0; flags[3] = max degree
__global__ void __launch_bounds__(256)
order_init_kernel(int64_t n, const int64_t* __restrict__ rank_nodes, const int32_t* __restrict__ degree,
                  int32_t* __restrict__ label, int32_t* __restrict__ node_of, uint64_t* __restrict__ owner,
                  uint8_t* __restrict__ visited, int32_t* __restrict__ flags) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int32_t d = 0;
  if (r < n) {
    const int64_t v = __ldg(rank_nodes + r);
    if (v < 0 || v >= n) {
      flags[2] = 1;
      node_of[r] = 0;
    } else {
      label[v] = (int32_t)r;
      node_of[r] = (int32_t)v;
      owner[v] = ~0ull;
      visited[v] = 0;
      d = __ldg(degree + v);
    }
  }
  d = __reduce_max_sync(0xffffffffu, d);
  if ((threadIdx.x & 31) == 0 && d > 0) atomicMax(flags + 3, d);
}

// rank_nodes is a permutation iff every node got a label (labels start at -1) that maps back to it
__global__ void __launch_bounds__(256)
order_check_kernel(int64_t n, const int32_t* __restrict__ label, const int32_t* __restrict__ node_of,
                   int32_t* __restrict__ flags) {
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= n) return;
  const int32_t l = label[v];
  if (l < 0 || l >= n || node_of[l] != (int32_t)v) flags[2] = 1;
}

// one warp per row u: an edge between two trees hooks the root of the larger label under the smaller one
__global__ void __launch_bounds__(256)
cc_hook_kernel(int64_t n, const int64_t* __restrict__ indptr, const int32_t* __restrict__ indices,
               const int32_t* __restrict__ node_of, int32_t* label, int32_t* __restrict__ changed) {
  const int64_t u = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (u >= n) return;
  const int64_t lo = __ldg(indptr + u), hi = __ldg(indptr + u + 1);
  for (int64_t e = lo + lane; e < hi; e += 32) {
    const int32_t a = label[u], b = label[__ldg(indices + e)];
    if (a == b) continue;
    const int32_t big = a > b ? a : b, small = a > b ? b : a;
    atomicMin(label + node_of[big], small);
    *changed = 1;
  }
}

// pointer jumping to the root: labels only decrease, a root (label == own rank) does not move here
__global__ void __launch_bounds__(256)
cc_jump_kernel(int64_t n, const int32_t* __restrict__ node_of, int32_t* label) {
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= n) return;
  int32_t l = label[v];
  for (;;) {
    const int32_t up = label[node_of[l]];
    if (up == l) break;
    l = up;
  }
  label[v] = l;
}

// ---- BFS ------------------------------------------------------------------------------------------------
// level 0: the seeds (label == own rank).  Their order is free: components are separated by the final
// stable sort, and the relative order of the nodes of one component never depends on the others.
__global__ void __launch_bounds__(256)
bfs_seed_kernel(int64_t n, const int32_t* __restrict__ node_of, const int32_t* __restrict__ label,
                int32_t* __restrict__ order, uint8_t* __restrict__ visited, int32_t* __restrict__ count) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int lane = threadIdx.x & 31;
  const int32_t v = r < n ? node_of[r] : 0;
  const bool seed = r < n && label[v] == (int32_t)r;
  const uint32_t ball = __ballot_sync(0xffffffffu, seed);
  int32_t at = 0;
  if (lane == 0 && ball) at = atomicAdd(count, __popc(ball));
  at = __shfl_sync(0xffffffffu, at, 0);
  if (seed) {
    order[at + __popc(ball & ((1u << lane) - 1))] = v;
    visited[v] = 1;
  }
}

// one warp per frontier position p: every unvisited neighbour takes the smallest (p, k) that reaches it
__global__ void __launch_bounds__(256)
bfs_elect_kernel(int64_t m, const int32_t* __restrict__ front, const int64_t* __restrict__ indptr,
                 const int32_t* __restrict__ indices, const uint8_t* __restrict__ visited,
                 unsigned long long* __restrict__ owner) {
  const int64_t p = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (p >= m) return;
  const int32_t u = front[p];
  const int64_t lo = __ldg(indptr + u), hi = __ldg(indptr + u + 1);
  for (int64_t e = lo + lane; e < hi; e += 32) {
    const int32_t j = __ldg(indices + e);
    if (!visited[j]) atomicMin(owner + j, ((unsigned long long)p << 32) | (unsigned long long)(e - lo));
  }
}

// winners of frontier position p (cnt[m] = 0 so that the scan's last item is the level size)
__global__ void __launch_bounds__(256)
bfs_count_kernel(int64_t m, const int32_t* __restrict__ front, const int64_t* __restrict__ indptr,
                 const int32_t* __restrict__ indices, const uint8_t* __restrict__ visited,
                 const uint64_t* __restrict__ owner, int32_t* __restrict__ cnt) {
  const int64_t p = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (p > m) return;
  if (p == m) {
    if (lane == 0) cnt[m] = 0;
    return;
  }
  const int32_t u = front[p];
  const int64_t lo = __ldg(indptr + u), hi = __ldg(indptr + u + 1);
  int32_t c = 0;
  for (int64_t b = lo; b < hi; b += 32) {
    const int64_t e = b + lane;
    bool win = false;
    if (e < hi) {
      const int32_t j = __ldg(indices + e);
      win = !visited[j] && owner[j] == (((uint64_t)p << 32) | (uint64_t)(e - lo));
    }
    c += __popc(__ballot_sync(0xffffffffu, win));
  }
  if (lane == 0) cnt[p] = c;
}

// the winners in (p, k) order at off[p] ..., keyed (p, degree) for the stable sort; marks them visited
__global__ void __launch_bounds__(256)
bfs_write_kernel(int64_t m, int dbits, const int32_t* __restrict__ front, const int64_t* __restrict__ indptr,
                 const int32_t* __restrict__ indices, const int32_t* __restrict__ degree, uint8_t* visited,
                 const uint64_t* __restrict__ owner, const int32_t* __restrict__ off, uint64_t* __restrict__ keys,
                 int32_t* __restrict__ vals) {
  const int64_t p = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (p >= m) return;
  const int32_t u = front[p];
  const int64_t lo = __ldg(indptr + u), hi = __ldg(indptr + u + 1);
  int64_t out = off[p];
  for (int64_t b = lo; b < hi; b += 32) {
    const int64_t e = b + lane;
    bool win = false;
    int32_t j = 0;
    if (e < hi) {
      j = __ldg(indices + e);
      // a node marked visited below belongs to this warp's own winners: no other (p, k) owns it
      win = !visited[j] && owner[j] == (((uint64_t)p << 32) | (uint64_t)(e - lo));
    }
    const uint32_t ball = __ballot_sync(0xffffffffu, win);
    if (win) {
      const int64_t at = out + __popc(ball & ((1u << lane) - 1));
      keys[at] = ((uint64_t)p << dbits) | (uint64_t)__ldg(degree + j);
      vals[at] = j;
      visited[j] = 1;
    }
    out += __popc(ball);
  }
}

// ---- order ----------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
order_key_kernel(int64_t n, const int32_t* __restrict__ order, const int32_t* __restrict__ label,
                 uint32_t* __restrict__ keys, int32_t* __restrict__ vals) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int32_t v = order[i];
  keys[i] = (uint32_t)label[v];
  vals[i] = v;
}

__global__ void __launch_bounds__(256)
order_reverse_kernel(int64_t n, const int32_t* __restrict__ sorted, int64_t* __restrict__ perm) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) perm[n - 1 - i] = sorted[i];
}

// ---- workspaces ------------------------------------------------------------------------------------------
struct RcmSymWs {
  uint64_t *keys_a, *keys_b;
  uint32_t *vals_a, *vals_b;
  int64_t* num_unique;
  int32_t* flags;   // [0] input not canonical, [1] id out of range
  void* cub_tmp;
  size_t cub_bytes, total;
};

RcmSymWs carve_rcm_sym(void* ws, int64_t n, int64_t nnz) {
  RcmSymWs w;
  Carver c{ws};
  const int64_t items = 2 * nnz > 0 ? 2 * nnz : 1;
  w.keys_a = (uint64_t*)c.take(sizeof(uint64_t) * (size_t)items);
  w.keys_b = (uint64_t*)c.take(sizeof(uint64_t) * (size_t)items);
  w.vals_a = (uint32_t*)c.take(sizeof(uint32_t) * (size_t)items);
  w.vals_b = (uint32_t*)c.take(sizeof(uint32_t) * (size_t)items);
  w.num_unique = (int64_t*)c.take(sizeof(int64_t));
  w.flags = (int32_t*)c.take(sizeof(int32_t) * 2);
  size_t sort_bytes = 0, uniq_bytes = 0;
  cub::DoubleBuffer<uint64_t> dk(nullptr, nullptr);
  cub::DoubleBuffer<uint32_t> dv(nullptr, nullptr);
  cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, dk, dv, items);
  cub::DeviceSelect::UniqueByKey(nullptr, uniq_bytes, (const uint64_t*)nullptr, (const uint32_t*)nullptr,
                                 (uint64_t*)nullptr, (uint32_t*)nullptr, (int64_t*)nullptr, items);
  w.cub_bytes = sort_bytes > uniq_bytes ? sort_bytes : uniq_bytes;
  w.cub_tmp = c.take(w.cub_bytes);
  w.total = c.off;
  return w;
}

struct OrderWs {
  int32_t *label, *node_of, *order, *cnt, *off, *vals_a, *vals_b;
  uint64_t *keys_a, *keys_b, *owner;
  uint32_t *fkeys_a, *fkeys_b;
  uint8_t* visited;
  int32_t* flags;   // [0] changed, [1] count, [2] rank_nodes not a permutation, [3] max degree
  void* cub_tmp;
  size_t cub_bytes, total;
};

OrderWs carve_order(void* ws, int64_t n) {
  OrderWs w;
  Carver c{ws};
  const size_t un = (size_t)n;
  w.label = (int32_t*)c.take(sizeof(int32_t) * un);
  w.node_of = (int32_t*)c.take(sizeof(int32_t) * un);
  w.order = (int32_t*)c.take(sizeof(int32_t) * un);
  w.cnt = (int32_t*)c.take(sizeof(int32_t) * (un + 1));
  w.off = (int32_t*)c.take(sizeof(int32_t) * (un + 1));
  w.vals_a = (int32_t*)c.take(sizeof(int32_t) * un);
  w.vals_b = (int32_t*)c.take(sizeof(int32_t) * un);
  w.keys_a = (uint64_t*)c.take(sizeof(uint64_t) * un);
  w.keys_b = (uint64_t*)c.take(sizeof(uint64_t) * un);
  w.owner = (uint64_t*)c.take(sizeof(uint64_t) * un);
  w.fkeys_a = (uint32_t*)c.take(sizeof(uint32_t) * un);
  w.fkeys_b = (uint32_t*)c.take(sizeof(uint32_t) * un);
  w.visited = (uint8_t*)c.take(un);
  w.flags = (int32_t*)c.take(sizeof(int32_t) * 4);
  size_t scan_bytes = 0, sort_bytes = 0, fsort_bytes = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, (const int32_t*)nullptr, (int32_t*)nullptr, n + 1);
  cub::DoubleBuffer<uint64_t> dk(nullptr, nullptr);
  cub::DoubleBuffer<uint32_t> fk(nullptr, nullptr);
  cub::DoubleBuffer<int32_t> dv(nullptr, nullptr);
  cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, dk, dv, n);
  cub::DeviceRadixSort::SortPairs(nullptr, fsort_bytes, fk, dv, n);
  w.cub_bytes = scan_bytes;
  if (sort_bytes > w.cub_bytes) w.cub_bytes = sort_bytes;
  if (fsort_bytes > w.cub_bytes) w.cub_bytes = fsort_bytes;
  w.cub_tmp = c.take(w.cub_bytes);
  w.total = c.off;
  return w;
}

double ms_since(std::chrono::steady_clock::time_point t0) {
  return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
}

}  // namespace
}  // namespace ttg

using namespace ttg;

extern "C" size_t ttg_rcm_symmetrise_workspace_bytes(int64_t num_nodes, int64_t num_edges) {
  if (!nodes_in_range(num_nodes) || !edges_in_range(num_edges)) return 0;
  return carve_rcm_sym(nullptr, num_nodes, num_edges).total;
}

extern "C" int ttg_rcm_symmetrise(int64_t num_nodes, int64_t num_edges, const int64_t* indptr,
                                  const int32_t* indices, int64_t* sym_indptr, int32_t* sym_indices,
                                  int32_t* degree, int64_t* sym_edges_out, void* workspace,
                                  size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  TTG_CHECK_ARG(nodes_in_range(num_nodes), "rcm_symmetrise: num_nodes=%lld out of range", (long long)num_nodes);
  TTG_CHECK_ARG(edges_in_range(num_edges), "rcm_symmetrise: num_edges=%lld out of range", (long long)num_edges);
  TTG_CHECK_ARG(indptr && (indices || num_edges == 0) && sym_indptr && sym_indices && degree && sym_edges_out,
                "rcm_symmetrise: null pointer");
  RcmSymWs w = carve_rcm_sym(workspace, num_nodes, num_edges);
  TTG_RC(check_workspace("rcm_symmetrise", workspace, workspace_bytes, w.total));
  const int colbits = bits_for((uint64_t)(num_nodes - 1));
  const int64_t items = 2 * num_edges;
  int64_t m = 0;
  int32_t flags[2] = {0, 0};
  TTG_CUDA(cudaMemsetAsync(w.flags, 0, 2 * sizeof(int32_t), stream));
  if (items > 0) {
    sym_emit_kernel<<<grid(num_nodes * 32), 256, 0, stream>>>(num_nodes, num_edges, colbits, indptr, indices,
                                                              w.keys_a, w.vals_a, w.flags);
    TTG_LAUNCH_CHECK();
    cub::DoubleBuffer<uint64_t> dk(w.keys_a, w.keys_b);
    cub::DoubleBuffer<uint32_t> dv(w.vals_a, w.vals_b);
    size_t bytes = w.cub_bytes;
    TTG_CUDA(cub::DeviceRadixSort::SortPairs(w.cub_tmp, bytes, dk, dv, items, 0, 2 * colbits, stream));
    count_launch();
    // the distinct pairs land in the other half of each double buffer
    uint64_t* ukeys = dk.Alternate();
    uint32_t* uvals = dv.Alternate();
    bytes = w.cub_bytes;
    TTG_CUDA(cub::DeviceSelect::UniqueByKey(w.cub_tmp, bytes, (const uint64_t*)dk.Current(),
                                            (const uint32_t*)dv.Current(), ukeys, uvals, w.num_unique, items,
                                            stream));
    count_launch();
    TTG_CUDA(cudaMemcpyAsync(flags, w.flags, sizeof(flags), cudaMemcpyDeviceToHost, stream));
    TTG_RC(read_back(&m, w.num_unique, stream));
    if (flags[1]) {
      set_error("rcm_symmetrise: an in-neighbour id lies outside [0, %lld) or indptr disagrees with num_edges",
                (long long)num_nodes);
      return TTG_EINVAL;
    }
    sym_rows_kernel<<<grid(num_nodes + 1), 256, 0, stream>>>(num_nodes, m, colbits, ukeys, sym_indptr, degree);
    TTG_LAUNCH_CHECK();
    if (m > 0 && !flags[0]) {   // canonical: rows are the sorted distinct columns already
      key_cols_kernel<<<grid(m), 256, 0, stream>>>(w.num_unique, (1ull << colbits) - 1, ukeys, sym_indices);
      TTG_LAUNCH_CHECK();
    } else if (m > 0) {        // general: each row in reverse order of first appearance
      uint64_t* rkeys = dk.Current();
      uint32_t* rcols = dv.Current();
      sym_reverse_key_kernel<<<grid(m), 256, 0, stream>>>(m, colbits, ukeys, uvals, rkeys, rcols);
      TTG_LAUNCH_CHECK();
      cub::DoubleBuffer<uint64_t> rk(rkeys, ukeys);
      cub::DoubleBuffer<uint32_t> rv(rcols, uvals);
      bytes = w.cub_bytes;
      TTG_CUDA(cub::DeviceRadixSort::SortPairs(w.cub_tmp, bytes, rk, rv, m, 0, 32 + colbits, stream));
      count_launch();
      TTG_CUDA(cudaMemcpyAsync(sym_indices, rv.Current(), sizeof(int32_t) * (size_t)m, cudaMemcpyDeviceToDevice,
                               stream));
    }
  } else {
    TTG_CUDA(cudaMemsetAsync(sym_indptr, 0, sizeof(int64_t) * (size_t)(num_nodes + 1), stream));
    TTG_CUDA(cudaMemsetAsync(degree, 0, sizeof(int32_t) * (size_t)num_nodes, stream));
  }
  *sym_edges_out = m;
  return TTG_OK;
}

extern "C" size_t ttg_rcm_order_workspace_bytes(int64_t num_nodes) {
  if (!nodes_in_range(num_nodes)) return 0;
  return carve_order(nullptr, num_nodes).total;
}

extern "C" int ttg_rcm_order(int64_t num_nodes, int64_t sym_edges, const int64_t* sym_indptr,
                             const int32_t* sym_indices, const int32_t* degree, const int64_t* rank_nodes,
                             int64_t* perm, int64_t* stats_out, double* phase_ms_out, void* workspace,
                             size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  TTG_CHECK_ARG(nodes_in_range(num_nodes), "rcm_order: num_nodes=%lld out of range", (long long)num_nodes);
  TTG_CHECK_ARG(sym_edges >= 0 && sym_edges <= 2 * kMaxEdges, "rcm_order: sym_edges=%lld out of range",
                (long long)sym_edges);
  TTG_CHECK_ARG(sym_indptr && (sym_indices || sym_edges == 0) && degree && rank_nodes && perm,
                "rcm_order: null pointer");
  OrderWs w = carve_order(workspace, num_nodes);
  TTG_RC(check_workspace("rcm_order", workspace, workspace_bytes, w.total));
  const int64_t n = num_nodes;
  const unsigned nb = grid(n);
  const auto t0 = std::chrono::steady_clock::now();

  // components: converged label = rank of the component's seed
  TTG_CUDA(cudaMemsetAsync(w.flags, 0, 4 * sizeof(int32_t), stream));
  TTG_CUDA(cudaMemsetAsync(w.label, 0xff, sizeof(int32_t) * (size_t)n, stream));
  order_init_kernel<<<nb, 256, 0, stream>>>(n, rank_nodes, degree, w.label, w.node_of, w.owner, w.visited,
                                            w.flags);
  TTG_LAUNCH_CHECK();
  order_check_kernel<<<nb, 256, 0, stream>>>(n, w.label, w.node_of, w.flags);
  TTG_LAUNCH_CHECK();
  int32_t flags[4];
  TTG_CUDA(cudaMemcpyAsync(flags, w.flags, sizeof(flags), cudaMemcpyDeviceToHost, stream));
  TTG_CUDA(cudaStreamSynchronize(stream));
  if (flags[2]) {
    set_error("rcm_order: rank_nodes is not a permutation of 0..%lld", (long long)n - 1);
    return TTG_EINVAL;
  }
  const int dbits = bits_for((uint64_t)flags[3]);
  if (sym_edges > 0) {
    for (int32_t changed = 1; changed;) {
      TTG_CUDA(cudaMemsetAsync(w.flags, 0, sizeof(int32_t), stream));
      cc_hook_kernel<<<grid(n * 32), 256, 0, stream>>>(n, sym_indptr, sym_indices, w.node_of, w.label, w.flags);
      TTG_LAUNCH_CHECK();
      cc_jump_kernel<<<nb, 256, 0, stream>>>(n, w.node_of, w.label);
      TTG_LAUNCH_CHECK();
      TTG_RC(read_back(&changed, w.flags, stream));
    }
  }
  const double t_cc = ms_since(t0);

  // BFS over every component at once; order[] collects the levels
  TTG_CUDA(cudaMemsetAsync(w.flags + 1, 0, sizeof(int32_t), stream));
  bfs_seed_kernel<<<nb, 256, 0, stream>>>(n, w.node_of, w.label, w.order, w.visited, w.flags + 1);
  TTG_LAUNCH_CHECK();
  int32_t components = 0;
  TTG_RC(read_back(&components, w.flags + 1, stream));
  int64_t front = 0, m = components, pos = components, levels = 1;
  while (m > 0 && sym_edges > 0) {
    const unsigned wb = grid(m * 32);
    bfs_elect_kernel<<<wb, 256, 0, stream>>>(m, w.order + front, sym_indptr, sym_indices, w.visited,
                                             (unsigned long long*)w.owner);
    TTG_LAUNCH_CHECK();
    bfs_count_kernel<<<grid((m + 1) * 32), 256, 0, stream>>>(m, w.order + front, sym_indptr, sym_indices, w.visited,
                                                             w.owner, w.cnt);
    TTG_LAUNCH_CHECK();
    size_t bytes = w.cub_bytes;
    TTG_CUDA(cub::DeviceScan::ExclusiveSum(w.cub_tmp, bytes, (const int32_t*)w.cnt, w.off, m + 1, stream));
    count_launch();
    int32_t next = 0;
    TTG_RC(read_back(&next, w.off + m, stream));
    if (next == 0) break;
    if (pos + next > n) {
      set_error("rcm_order: BFS level overflows %lld nodes (sym lists inconsistent)", (long long)n);
      return TTG_EINVAL;
    }
    bfs_write_kernel<<<wb, 256, 0, stream>>>(m, dbits, w.order + front, sym_indptr, sym_indices, degree,
                                             w.visited, w.owner, w.off, w.keys_a, w.vals_a);
    TTG_LAUNCH_CHECK();
    cub::DoubleBuffer<uint64_t> dk(w.keys_a, w.keys_b);
    cub::DoubleBuffer<int32_t> dv(w.vals_a, w.vals_b);
    bytes = w.cub_bytes;
    TTG_CUDA(cub::DeviceRadixSort::SortPairs(w.cub_tmp, bytes, dk, dv, (int64_t)next, 0,
                                             bits_for((uint64_t)(m - 1)) + dbits, stream));
    count_launch();
    TTG_CUDA(cudaMemcpyAsync(w.order + pos, dv.Current(), sizeof(int32_t) * (size_t)next,
                             cudaMemcpyDeviceToDevice, stream));
    front = pos;
    pos += next;
    m = next;
    ++levels;
  }
  const double t_bfs = ms_since(t0) - t_cc;
  if (pos != n) {
    set_error("rcm_order: the BFS reached %lld of %lld nodes (sym lists not symmetric?)", (long long)pos,
              (long long)n);
    return TTG_EINVAL;
  }

  // components in seed-rank order (stable: each keeps its level order), then reversed
  order_key_kernel<<<nb, 256, 0, stream>>>(n, w.order, w.label, w.fkeys_a, w.vals_a);
  TTG_LAUNCH_CHECK();
  cub::DoubleBuffer<uint32_t> fk(w.fkeys_a, w.fkeys_b);
  cub::DoubleBuffer<int32_t> fv(w.vals_a, w.vals_b);
  size_t bytes = w.cub_bytes;
  TTG_CUDA(cub::DeviceRadixSort::SortPairs(w.cub_tmp, bytes, fk, fv, n, 0, bits_for((uint64_t)(n - 1)), stream));
  count_launch();
  order_reverse_kernel<<<nb, 256, 0, stream>>>(n, fv.Current(), perm);
  TTG_LAUNCH_CHECK();
  if (stats_out) {
    stats_out[0] = levels;
    stats_out[1] = components;
  }
  if (phase_ms_out) {
    TTG_CUDA(cudaStreamSynchronize(stream));
    phase_ms_out[0] = t_cc;
    phase_ms_out[1] = t_bfs;
    phase_ms_out[2] = ms_since(t0) - t_cc - t_bfs;
  }
  return TTG_OK;
}
