// reorder.cu -- node reordering of a CSR graph on the device (SURVEY 8f-3).
//
// The reference renumbers the nodes before training so that the ids a minibatch touches share
// TT prefixes and cache lines: dgl.reorder_graph(graph, 'metis' | 'rcmk' | 'custom')
// (graphloader.py:358-372, 399-454; DGL 2.1 and METIS are un-vendored).  Two pieces live here:
//
//   permute   the graph under a node permutation (new node n = old node perm[n], DGL's
//             nodes_perm convention): degrees gathered -> exclusive scan -> every in-neighbour list
//             copied in its old order with the ids mapped through the inverse permutation.
//             Integer work, bit-exact against oracle/reorder_oracle.py.
//   grow      a k-way partition grown from k seed nodes by capacity-bounded label propagation
//             (a node takes the part of the first in-neighbour whose part still has room), the
//             stand-in for METIS-k where METIS is not available.  It is NOT METIS: the parts are
//             connected and bounded in size, the cut is whatever the growth leaves.  The result
//             depends on the order in which parts fill up (atomics), so only its invariants are
//             tested.  RCMK: DGL calls scipy.sparse.csgraph.reverse_cuthill_mckee and so does
//             reorder.py by default; csrc/rcm.cu computes the same permutation on the device
//             (reorder_graph(g, "rcmk", backend="device")).
#include <cub/device/device_scan.cuh>

#include "graph.cuh"

namespace ttg {
namespace {

constexpr int32_t kBadPerm = 1, kBadGraph = 2;   // the bits of bad_flag (ttg_b200.h)

// new row i = old row perm[i]: its length, checked, and inv[perm[i]] = i
__global__ void __launch_bounds__(256)
perm_degree_kernel(int64_t n, const int64_t* __restrict__ indptr, const int64_t* __restrict__ perm,
                   int64_t* __restrict__ inv, int64_t* __restrict__ deg, int32_t* __restrict__ bad) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i > n) return;
  if (i == n) {
    deg[n] = 0;   // the scan runs over n + 1 items so that new_indptr[n] comes out of it
    return;
  }
  const int64_t old = __ldg(perm + i);
  if (old < 0 || old >= n) {
    atomicOr(bad, kBadPerm);
    deg[i] = 0;
    return;
  }
  inv[old] = i;
  int64_t lo, hi;
  const bool ok = csr_row(indptr, n, __ldg(indptr + n), old, &lo, &hi);
  if (!ok) atomicOr(bad, kBadGraph);
  deg[i] = ok ? hi - lo : 0;
}

// one warp per new row
__global__ void __launch_bounds__(256)
perm_fill_kernel(int64_t n, const int64_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                 const int64_t* __restrict__ perm, const int64_t* __restrict__ inv,
                 const int64_t* __restrict__ new_indptr, int32_t* __restrict__ new_indices, int32_t* bad) {
  const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= n || *bad) return;   // every row read below passed perm_degree_kernel's checks
  const int64_t old = __ldg(perm + row);
  const int64_t src = __ldg(indptr + old), cnt = __ldg(indptr + old + 1) - src;
  const int64_t dst = __ldg(new_indptr + row);
  bool out = false;   // an id outside [0, n): reported once after the loop, which stays free of atomics
  for (int64_t j = lane; j < cnt; j += 32) {
    const int32_t u = __ldg(indices + src + j);
    const bool in = u >= 0 && u < n;
    out |= !in;
    new_indices[dst + j] = (int32_t)__ldg(inv + (in ? u : 0));
  }
  if (out) atomicOr(bad, kBadGraph);
}

__global__ void __launch_bounds__(256)
grow_init_kernel(int64_t n, int32_t k, const int64_t* __restrict__ seeds, int32_t* __restrict__ labels,
                 int32_t* __restrict__ sizes) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) labels[i] = -1;
  if (i < k) sizes[i] = 0;
}
__global__ void __launch_bounds__(256)
grow_seed_kernel(int64_t n, int32_t k, const int64_t* __restrict__ seeds, int32_t* __restrict__ labels,
                 int32_t* __restrict__ sizes) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= k) return;
  const int64_t s = __ldg(seeds + i);
  if (s < 0 || s >= n) return;
  if (atomicCAS(labels + s, -1, i) == -1) atomicAdd(sizes + i, 1);   // duplicate seeds: first wins
}

// one sweep: every unlabelled node looks at the labels its in-neighbours had BEFORE the sweep
__global__ void __launch_bounds__(256)
grow_sweep_kernel(int64_t n, const int64_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                  int32_t cap, const int32_t* __restrict__ labels_in, int32_t* __restrict__ labels_out,
                  int32_t* __restrict__ sizes, int32_t* __restrict__ changed) {
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= n) return;
  int32_t l = labels_in[v];
  if (l < 0) {
    const int64_t lo = __ldg(indptr + v), hi = __ldg(indptr + v + 1);
    for (int64_t e = lo; e < hi; ++e) {
      const int32_t c = labels_in[__ldg(indices + e)];
      if (c < 0) continue;
      if (atomicAdd(sizes + c, 1) < cap) {
        l = c;
        *changed = 1;
        break;
      }
      atomicSub(sizes + c, 1);   // full: try the next neighbour's part
    }
  }
  labels_out[v] = l;
}

}  // namespace
}  // namespace ttg

using namespace ttg;

namespace {
struct PermWs {
  int64_t* inv;
  int64_t* deg;
  int32_t* bad;
  void* cub_tmp;
  size_t cub_bytes, total;
};
PermWs carve_perm(void* ws, int64_t n) {
  PermWs w;
  Carver c{ws};
  w.inv = (int64_t*)c.take(sizeof(int64_t) * (size_t)n);
  w.deg = (int64_t*)c.take(sizeof(int64_t) * (size_t)(n + 1));
  w.bad = (int32_t*)c.take(sizeof(int32_t));
  w.cub_bytes = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, w.cub_bytes, (const int64_t*)nullptr, (int64_t*)nullptr, (int)(n + 1));
  w.cub_tmp = c.take(w.cub_bytes);
  w.total = c.off;
  return w;
}
}  // namespace

extern "C" size_t ttg_permute_csr_workspace_bytes(int64_t num_nodes) {
  if (!nodes_in_range(num_nodes)) return 0;
  return carve_perm(nullptr, num_nodes).total;
}

extern "C" int ttg_permute_csr(int64_t num_nodes, const int64_t* indptr, const int32_t* indices,
                               const int64_t* perm, int64_t* new_indptr, int32_t* new_indices,
                               int64_t* inverse_out, int32_t* bad_flag, void* workspace,
                               size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  TTG_CHECK_ARG(nodes_in_range(num_nodes), "permute_csr: num_nodes=%lld out of range", (long long)num_nodes);
  TTG_CHECK_ARG(indptr && perm && new_indptr && bad_flag, "permute_csr: null pointer");
  PermWs w = carve_perm(workspace, num_nodes);
  TTG_RC(check_workspace("permute_csr", workspace, workspace_bytes, w.total));
  int64_t* inv = inverse_out ? inverse_out : w.inv;
  TTG_CUDA(cudaMemsetAsync(bad_flag, 0, sizeof(int32_t), stream));
  perm_degree_kernel<<<grid(num_nodes + 1), 256, 0, stream>>>(num_nodes, indptr, perm, inv, w.deg, bad_flag);
  TTG_LAUNCH_CHECK();
  size_t bytes = w.cub_bytes;
  TTG_CUDA(cub::DeviceScan::ExclusiveSum(w.cub_tmp, bytes, (const int64_t*)w.deg, new_indptr,
                                         (int)(num_nodes + 1), stream));
  count_launch();
  perm_fill_kernel<<<grid(num_nodes * 32), 256, 0, stream>>>(num_nodes, indptr, indices, perm, inv, new_indptr,
                                                             new_indices, bad_flag);
  TTG_LAUNCH_CHECK();
  return TTG_OK;
}

/* labels_a / labels_b: two int32 [num_nodes] buffers (the sweeps ping-pong between them; the
 * result is in labels_a), sizes int32 [k], changed int32 [1].  `sweeps` must be even. */
extern "C" int ttg_partition_grow(int64_t num_nodes, const int64_t* indptr, const int32_t* indices,
                                  int32_t k, int32_t cap, const int64_t* seeds, int32_t sweeps,
                                  int32_t* labels_a, int32_t* labels_b, int32_t* sizes,
                                  int32_t* changed, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  TTG_CHECK_ARG(num_nodes > 0 && k > 0 && cap > 0 && sweeps > 0 && sweeps % 2 == 0,
                "partition_grow: bad sizes (nodes %lld, k %d, cap %d, sweeps %d)", (long long)num_nodes,
                k, cap, sweeps);
  TTG_CHECK_ARG((int64_t)k * cap >= num_nodes, "partition_grow: k * cap = %lld < %lld nodes",
                (long long)k * cap, (long long)num_nodes);
  TTG_CHECK_ARG(indptr && labels_a && labels_b && sizes && changed, "partition_grow: null pointer");
  if (seeds) {   // first call: start from the seeds; later calls (seeds == NULL) continue from labels_a
    const unsigned nb = grid(num_nodes > k ? num_nodes : k);
    grow_init_kernel<<<nb, 256, 0, stream>>>(num_nodes, k, seeds, labels_a, sizes);
    TTG_LAUNCH_CHECK();
    grow_seed_kernel<<<grid(k), 256, 0, stream>>>(num_nodes, k, seeds, labels_a, sizes);
    TTG_LAUNCH_CHECK();
  }
  TTG_CUDA(cudaMemsetAsync(changed, 0, sizeof(int32_t), stream));
  for (int s = 0; s < sweeps; ++s) {
    grow_sweep_kernel<<<grid(num_nodes), 256, 0, stream>>>(
        num_nodes, indptr, indices, cap, (s & 1) ? labels_b : labels_a, (s & 1) ? labels_a : labels_b,
        sizes, changed);
    TTG_LAUNCH_CHECK();
  }
  return TTG_OK;
}
