// spmm.cu -- neighbour aggregation on a sampled block: CSR (by destination) SpMM.
//
// Replaces the SpMM inside dglnn.SAGEConv(..., 'mean') (gnn_model.py:78-81, called :211-214)
// and the sum aggregation of dglnn.GraphConv(norm='both') (gnn_model.py:287); DGL 2.1.0 is not
// vendored in the reference, the semantics restated in oracle/ are:
//   out[v] = scale_v * sum_{e in N_in(v)} w_e * x[src(e)],   mean: scale_v = 1/deg(v) (0 if none)
// HBM-bound gather: one warp per destination row, 16-byte loads of the source rows, edges
// unrolled by four so four independent row gathers are in flight per lane.
#include <cub/cub.cuh>

#include "common.cuh"

namespace ttg {
namespace {

__global__ void __launch_bounds__(256)
spmm_fwd_kernel(int64_t num_dst, int32_t F, const int64_t* __restrict__ indptr,
                const int32_t* __restrict__ indices, const float* __restrict__ ew, int mean,
                const float* __restrict__ x, float* __restrict__ out) {
  const int64_t v = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (v >= num_dst) return;
  const int64_t e0 = __ldg(indptr + v), e1 = __ldg(indptr + v + 1);
  const float scale = (mean && e1 > e0) ? 1.0f / (float)(e1 - e0) : 1.0f;
  for (int d = lane * 4; d < F; d += 128) {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    int64_t e = e0;
    for (; e + 4 <= e1; e += 4) {
      int32_t s[4];
      float w[4];
      float4 r[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        s[u] = __ldg(indices + e + u);
        w[u] = ew ? __ldg(ew + e + u) : 1.0f;
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) r[u] = ldg4(x + (int64_t)s[u] * F + d);
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        acc.x = fmaf(w[u], r[u].x, acc.x);
        acc.y = fmaf(w[u], r[u].y, acc.y);
        acc.z = fmaf(w[u], r[u].z, acc.z);
        acc.w = fmaf(w[u], r[u].w, acc.w);
      }
    }
    for (; e < e1; ++e) {
      const int32_t s = __ldg(indices + e);
      const float w = ew ? __ldg(ew + e) : 1.0f;
      const float4 r = ldg4(x + (int64_t)s * F + d);
      acc.x = fmaf(w, r.x, acc.x);
      acc.y = fmaf(w, r.y, acc.y);
      acc.z = fmaf(w, r.z, acc.z);
      acc.w = fmaf(w, r.w, acc.w);
    }
    acc.x *= scale;
    acc.y *= scale;
    acc.z *= scale;
    acc.w *= scale;
    *reinterpret_cast<float4*>(out + v * F + d) = acc;
  }
}

__global__ void __launch_bounds__(256)
spmm_bwd_kernel(int64_t num_dst, int32_t F, const int64_t* __restrict__ indptr,
                const int32_t* __restrict__ indices, const float* __restrict__ ew, int mean,
                const float* __restrict__ dout, float* __restrict__ dx) {
  const int64_t v = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (v >= num_dst) return;
  const int64_t e0 = __ldg(indptr + v), e1 = __ldg(indptr + v + 1);
  if (e1 <= e0) return;
  const float scale = mean ? 1.0f / (float)(e1 - e0) : 1.0f;
  for (int d = lane * 4; d < F; d += 128) {
    float4 g = ldg4(dout + v * F + d);
    g.x *= scale;
    g.y *= scale;
    g.z *= scale;
    g.w *= scale;
    for (int64_t e = e0; e < e1; ++e) {
      const int32_t s = __ldg(indices + e);
      const float w = ew ? __ldg(ew + e) : 1.0f;
      red_add_v4(dx + (int64_t)s * F + d, make_float4(w * g.x, w * g.y, w * g.z, w * g.w));
    }
  }
}

// rows whose width is not a multiple of four floats (the 47-class output layer): scalar lanes
__global__ void __launch_bounds__(256)
spmm_fwd_scalar_kernel(int64_t num_dst, int32_t F, const int64_t* __restrict__ indptr,
                       const int32_t* __restrict__ indices, const float* __restrict__ ew, int mean,
                       const float* __restrict__ x, float* __restrict__ out) {
  const int64_t v = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (v >= num_dst) return;
  const int64_t e0 = __ldg(indptr + v), e1 = __ldg(indptr + v + 1);
  const float scale = (mean && e1 > e0) ? 1.0f / (float)(e1 - e0) : 1.0f;
  for (int d = lane; d < F; d += 32) {
    float acc = 0.f;
    for (int64_t e = e0; e < e1; ++e) {
      const float w = ew ? __ldg(ew + e) : 1.0f;
      acc = fmaf(w, __ldg(x + (int64_t)__ldg(indices + e) * F + d), acc);
    }
    out[v * F + d] = acc * scale;
  }
}

__global__ void __launch_bounds__(256)
spmm_bwd_scalar_kernel(int64_t num_dst, int32_t F, const int64_t* __restrict__ indptr,
                       const int32_t* __restrict__ indices, const float* __restrict__ ew, int mean,
                       const float* __restrict__ dout, float* __restrict__ dx) {
  const int64_t v = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (v >= num_dst) return;
  const int64_t e0 = __ldg(indptr + v), e1 = __ldg(indptr + v + 1);
  if (e1 <= e0) return;
  const float scale = mean ? 1.0f / (float)(e1 - e0) : 1.0f;
  for (int d = lane; d < F; d += 32) {
    const float g = __ldg(dout + v * F + d) * scale;
    for (int64_t e = e0; e < e1; ++e) {
      const float w = ew ? __ldg(ew + e) : 1.0f;
      atomicAdd(dx + (int64_t)__ldg(indices + e) * F + d, w * g);
    }
  }
}

// ---- whole-graph mean aggregation, balanced by edges ------------------------------------------------
// The kernels above give one warp to each destination: right for sampled blocks (in-degree <= fanout <= 32),
// wrong for a whole power-law graph, where one warp would walk a row of 40 k edges alone.  Here every row
// is cut into work items of at most kAggW edges and a warp takes one item.  A node's only item writes its
// output row; the items of a longer row write one partial row each, which a second pass sums in item order
// and scales (deterministic, no float atomics).  The item list (the plan) depends on indptr alone.
constexpr int64_t kAggW = 256;   // edges per work item
constexpr int kAggU = 8;         // edges in flight per lane

struct AggItem {
  int64_t ebeg;   // first edge of the item; it ends at min(ebeg + kAggW, indptr[dst + 1])
  int32_t dst;
  int32_t slot;   // partial row of the item, -1: the node's only item (writes the output row)
};
struct AggCount {
  long long items, multi;   // work items of a node, 1 if it has more than one
};
struct AggCountSum {
  __host__ __device__ AggCount operator()(const AggCount& a, const AggCount& b) const {
    return AggCount{a.items + b.items, a.multi + b.multi};
  }
};

__host__ __device__ inline int64_t agg_items_of(int64_t deg) { return deg <= kAggW ? 1 : (deg + kAggW - 1) / kAggW; }

// bounds the host knows without looking at the graph: sum over nodes of max(1, ceil(d / W)) <= N + E / W;
// at most E / (W + 1) nodes have more than W edges, and their items number at most E / W + E / (W + 1)
int64_t agg_cap_items(int64_t n, int64_t e) { return n + e / kAggW; }
int64_t agg_cap_multi(int64_t e) { return e / (kAggW + 1); }
int64_t agg_cap_parts(int64_t e) { return e / kAggW + e / (kAggW + 1); }

struct AggPlan {        // carved from the caller's plan buffer
  int64_t* header;      // [2] {items, nodes with several items}
  AggItem* items;       // [cap_items]
  int64_t* multi;       // [cap_multi][2] {node, first partial row}
  size_t total;
};
AggPlan carve_agg_plan(void* base, int64_t n, int64_t e) {
  AggPlan p;
  size_t off = 0;
  char* b = (char*)base;
  p.header = (int64_t*)(b + off);
  off = align_up(off + 4 * sizeof(int64_t), 256);
  p.items = (AggItem*)(b + off);
  off = align_up(off + sizeof(AggItem) * (size_t)agg_cap_items(n, e), 256);
  p.multi = (int64_t*)(b + off);
  off = align_up(off + 2 * sizeof(int64_t) * (size_t)(agg_cap_multi(e) > 0 ? agg_cap_multi(e) : 1), 256);
  p.total = off;
  return p;
}

struct AggBuildWs {
  AggCount *count, *start;   // [n] per node, exclusive scan
  void* cub_tmp;
  size_t cub_bytes, total;
};
AggBuildWs carve_agg_build(void* base, int64_t n) {
  AggBuildWs w;
  size_t off = 0;
  char* b = (char*)base;
  const size_t m = (size_t)(n > 0 ? n : 1);
  w.count = (AggCount*)(b + off);
  off = align_up(off + sizeof(AggCount) * m, 256);
  w.start = (AggCount*)(b + off);
  off = align_up(off + sizeof(AggCount) * m, 256);
  w.cub_bytes = 0;
  cub::DeviceScan::ExclusiveScan(nullptr, w.cub_bytes, (const AggCount*)nullptr, (AggCount*)nullptr, AggCountSum(),
                                 AggCount{0, 0}, (int64_t)m, (cudaStream_t)0);
  w.cub_tmp = b + off;
  off = align_up(off + w.cub_bytes, 256);
  w.total = off;
  return w;
}
size_t agg_parts_bytes(int64_t e, int32_t F) {
  return align_up(sizeof(float) * (size_t)agg_cap_parts(e) * (size_t)F, 256) + 256;
}

__global__ void __launch_bounds__(256)
agg_count_kernel(int64_t n, const int64_t* __restrict__ indptr, AggCount* __restrict__ count) {
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= n) return;
  const int64_t k = agg_items_of(__ldg(indptr + v + 1) - __ldg(indptr + v));
  count[v] = AggCount{k, k > 1 ? 1 : 0};
}

__global__ void __launch_bounds__(256)
agg_scatter_kernel(int64_t n, const int64_t* __restrict__ indptr, const AggCount* __restrict__ start,
                   int64_t* __restrict__ header, AggItem* __restrict__ items, int64_t* __restrict__ multi) {
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= n) return;
  const int64_t rb = __ldg(indptr + v);
  const int64_t k = agg_items_of(__ldg(indptr + v + 1) - rb);
  const AggCount s = start[v];
  if (k == 1) {
    items[s.items] = AggItem{rb, (int32_t)v, -1};
  } else {
    // partial rows are numbered over the nodes with several items: items before v minus single-item nodes before v
    const int64_t first = s.items - (v - s.multi);
    for (int64_t j = 0; j < k; ++j) items[s.items + j] = AggItem{rb + j * kAggW, (int32_t)v, (int32_t)(first + j)};
    multi[2 * s.multi] = v;
    multi[2 * s.multi + 1] = first;
  }
  if (v == n - 1) {
    header[0] = s.items + k;
    header[1] = s.multi + (k > 1 ? 1 : 0);
  }
}

// One warp per item.  The item's indices are read once per 32 edges (one per lane) and handed round by
// shuffles; kAggU source rows are then loaded per lane and column before any is summed.  VEC: 16-byte
// columns (F % 4 == 0), else scalar ones; C column groups of the warp per pass over the edges.
template <int C, bool VEC>
__global__ void __launch_bounds__(256)
mean_agg_kernel(int64_t cap, int32_t F, const int64_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                const int64_t* __restrict__ header, const AggItem* __restrict__ items, const float* __restrict__ x,
                float* __restrict__ out, float* __restrict__ partial) {
  const int64_t it = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (it >= cap || it >= __ldg(header)) return;
  const int4 raw = __ldg(reinterpret_cast<const int4*>(items + it));
  const int64_t e0 = (int64_t)(((uint64_t)(uint32_t)raw.y << 32) | (uint32_t)raw.x);
  const int32_t v = raw.z, slot = raw.w;
  const int64_t rb = __ldg(indptr + v), re = __ldg(indptr + v + 1);
  const int64_t e1 = min(e0 + kAggW, re);
  float* dst;
  float scale;
  if (slot < 0) {
    dst = out + (int64_t)v * F;
    scale = re > rb ? 1.0f / (float)(re - rb) : 0.0f;
  } else {
    dst = partial + (int64_t)slot * F;
    scale = 1.0f;
  }
  constexpr int kLane = VEC ? 4 : 1;              // floats per lane and column group
  constexpr int kStep = 32 * kLane * C;           // columns per pass
  for (int d0 = 0; d0 < F; d0 += kStep) {
    float acc[C][kLane];
#pragma unroll
    for (int c = 0; c < C; ++c)
#pragma unroll
      for (int k = 0; k < kLane; ++k) acc[c][k] = 0.f;
    int col[C];
#pragma unroll
    for (int c = 0; c < C; ++c) col[c] = d0 + (c * 32 + lane) * kLane;
    for (int64_t base = e0; base < e1; base += 32) {
      const int n = (int)min((int64_t)32, e1 - base);
      const int32_t mine = lane < n ? __ldg(indices + base + lane) : 0;
      int j = 0;
      for (; j + kAggU <= n; j += kAggU) {
        float r[kAggU][C][kLane];
#pragma unroll
        for (int u = 0; u < kAggU; ++u) {
          const float* row = x + (int64_t)__shfl_sync(0xffffffffu, mine, j + u) * F;
#pragma unroll
          for (int c = 0; c < C; ++c) {
            if (col[c] < F) {
              if constexpr (VEC) {
                const float4 q = ldg4(row + col[c]);
                r[u][c][0] = q.x; r[u][c][1] = q.y; r[u][c][2] = q.z; r[u][c][3] = q.w;
              } else {
                r[u][c][0] = __ldg(row + col[c]);
              }
            } else {
#pragma unroll
              for (int k = 0; k < kLane; ++k) r[u][c][k] = 0.f;
            }
          }
        }
#pragma unroll
        for (int u = 0; u < kAggU; ++u)
#pragma unroll
          for (int c = 0; c < C; ++c)
#pragma unroll
            for (int k = 0; k < kLane; ++k) acc[c][k] += r[u][c][k];
      }
      for (; j < n; ++j) {
        const float* row = x + (int64_t)__shfl_sync(0xffffffffu, mine, j) * F;
#pragma unroll
        for (int c = 0; c < C; ++c) {
          if (col[c] < F) {
            if constexpr (VEC) {
              const float4 q = ldg4(row + col[c]);
              acc[c][0] += q.x; acc[c][1] += q.y; acc[c][2] += q.z; acc[c][3] += q.w;
            } else {
              acc[c][0] += __ldg(row + col[c]);
            }
          }
        }
      }
    }
#pragma unroll
    for (int c = 0; c < C; ++c) {
      if (col[c] < F) {
        if constexpr (VEC) {
          *reinterpret_cast<float4*>(dst + col[c]) =
              make_float4(acc[c][0] * scale, acc[c][1] * scale, acc[c][2] * scale, acc[c][3] * scale);
        } else {
          dst[col[c]] = acc[c][0] * scale;
        }
      }
    }
  }
}

// out row of every node with several items: its partial rows summed in item order, times 1 / deg
template <bool VEC>
__global__ void __launch_bounds__(256)
mean_agg_finalize_kernel(int64_t cap, int32_t F, const int64_t* __restrict__ indptr,
                         const int64_t* __restrict__ header, const int64_t* __restrict__ multi,
                         const float* __restrict__ partial, float* __restrict__ out) {
  const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (w >= cap || w >= __ldg(header + 1)) return;
  const int64_t v = __ldg(multi + 2 * w), first = __ldg(multi + 2 * w + 1);
  const int64_t deg = __ldg(indptr + v + 1) - __ldg(indptr + v);
  const int64_t k = agg_items_of(deg);
  const float scale = 1.0f / (float)deg;
  const float* p = partial + first * F;
  if constexpr (VEC) {
    for (int d = lane * 4; d < F; d += 128) {
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int64_t j = 0; j < k; ++j) {
        const float4 q = ldg4(p + j * F + d);
        acc.x += q.x; acc.y += q.y; acc.z += q.z; acc.w += q.w;
      }
      *reinterpret_cast<float4*>(out + v * F + d) =
          make_float4(acc.x * scale, acc.y * scale, acc.z * scale, acc.w * scale);
    }
  } else {
    for (int d = lane; d < F; d += 32) {
      float acc = 0.f;
      for (int64_t j = 0; j < k; ++j) acc += __ldg(p + j * F + d);
      out[v * F + d] = acc * scale;
    }
  }
}

bool agg_nodes_ok(int64_t n) { return n >= 0 && n < ((int64_t)1 << 31); }
// partial-row numbers are int32: E / W + E / (W + 1) < 2^31
bool agg_edges_ok(int64_t e) { return e >= 0 && e <= ((int64_t)1 << 37); }

}  // namespace
}  // namespace ttg

using namespace ttg;

extern "C" size_t ttg_mean_agg_plan_bytes(int64_t num_nodes, int64_t num_edges) {
  if (!agg_nodes_ok(num_nodes) || !agg_edges_ok(num_edges)) return 0;
  return carve_agg_plan(nullptr, num_nodes, num_edges).total;
}

extern "C" size_t ttg_mean_agg_workspace_bytes(int64_t num_nodes, int64_t num_edges, int32_t F) {
  if (!agg_nodes_ok(num_nodes) || !agg_edges_ok(num_edges) || F <= 0) return 0;
  const size_t build = carve_agg_build(nullptr, num_nodes).total;
  const size_t parts = agg_parts_bytes(num_edges, F);
  return build > parts ? build : parts;
}

extern "C" int ttg_mean_agg_plan(int64_t num_nodes, int64_t num_edges, const int64_t* indptr, void* plan,
                                 size_t plan_bytes, void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  TTG_CHECK_ARG(agg_nodes_ok(num_nodes), "mean_agg_plan: num_nodes=%lld out of range", (long long)num_nodes);
  TTG_CHECK_ARG(agg_edges_ok(num_edges), "mean_agg_plan: num_edges=%lld out of range", (long long)num_edges);
  TTG_CHECK_ARG(indptr && plan, "mean_agg_plan: null pointer");
  TTG_CHECK_ARG(((uintptr_t)plan & 15) == 0, "mean_agg_plan: plan buffer not 16-byte aligned");
  const AggPlan p = carve_agg_plan(plan, num_nodes, num_edges);
  if (plan_bytes < p.total) {
    set_error("mean_agg_plan: plan buffer %zu bytes, need %zu", plan_bytes, p.total);
    return TTG_ENOMEM;
  }
  const AggBuildWs w = carve_agg_build(workspace, num_nodes);
  if (!workspace || workspace_bytes < w.total) {
    set_error("mean_agg_plan: workspace %zu bytes, need %zu", workspace_bytes, w.total);
    return TTG_ENOMEM;
  }
  TTG_CUDA(cudaMemsetAsync(p.header, 0, 4 * sizeof(int64_t), stream));
  if (num_nodes == 0) return TTG_OK;
  const unsigned nb = (unsigned)ceil_div(num_nodes, 256);
  agg_count_kernel<<<nb, 256, 0, stream>>>(num_nodes, indptr, w.count);
  TTG_LAUNCH_CHECK();
  size_t bytes = w.cub_bytes;
  TTG_CUDA(cub::DeviceScan::ExclusiveScan(w.cub_tmp, bytes, (const AggCount*)w.count, w.start, AggCountSum(),
                                          AggCount{0, 0}, num_nodes, stream));
  count_launch();
  agg_scatter_kernel<<<nb, 256, 0, stream>>>(num_nodes, indptr, w.start, p.header, p.items, p.multi);
  TTG_LAUNCH_CHECK();
  return TTG_OK;
}

extern "C" int ttg_mean_agg(int64_t num_nodes, int64_t num_edges, int32_t F, const int64_t* indptr,
                            const int32_t* indices, const void* plan, size_t plan_bytes, const float* x,
                            float* out, void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  TTG_CHECK_ARG(F > 0, "mean_agg: F=%d must be positive", F);
  TTG_CHECK_ARG(agg_nodes_ok(num_nodes), "mean_agg: num_nodes=%lld out of range", (long long)num_nodes);
  TTG_CHECK_ARG(agg_edges_ok(num_edges), "mean_agg: num_edges=%lld out of range", (long long)num_edges);
  TTG_CHECK_ARG(indptr && (indices || num_edges == 0) && plan && x && out, "mean_agg: null pointer");
  TTG_CHECK_ARG(((uintptr_t)plan & 15) == 0, "mean_agg: plan buffer not 16-byte aligned");
  const AggPlan p = carve_agg_plan(const_cast<void*>(plan), num_nodes, num_edges);
  if (plan_bytes < p.total) {
    set_error("mean_agg: plan buffer %zu bytes, need %zu", plan_bytes, p.total);
    return TTG_ENOMEM;
  }
  const size_t need = ttg_mean_agg_workspace_bytes(num_nodes, num_edges, F);
  if (!workspace || workspace_bytes < need) {
    set_error("mean_agg: workspace %zu bytes, need %zu", workspace_bytes, need);
    return TTG_ENOMEM;
  }
  if (num_nodes == 0) return TTG_OK;
  float* partial = (float*)align_up((size_t)workspace, 256);
  const bool vec = F % 4 == 0 && (((uintptr_t)x | (uintptr_t)out) & 15) == 0;
  const int64_t cap = agg_cap_items(num_nodes, num_edges);
  const unsigned nb = (unsigned)ceil_div(cap * 32, 256);
  if (vec && F <= 128) {
    mean_agg_kernel<1, true><<<nb, 256, 0, stream>>>(cap, F, indptr, indices, p.header, p.items, x, out, partial);
  } else if (vec) {
    mean_agg_kernel<2, true><<<nb, 256, 0, stream>>>(cap, F, indptr, indices, p.header, p.items, x, out, partial);
  } else if (F <= 32) {
    mean_agg_kernel<1, false><<<nb, 256, 0, stream>>>(cap, F, indptr, indices, p.header, p.items, x, out, partial);
  } else {
    mean_agg_kernel<2, false><<<nb, 256, 0, stream>>>(cap, F, indptr, indices, p.header, p.items, x, out, partial);
  }
  TTG_LAUNCH_CHECK();
  const int64_t cap_multi = agg_cap_multi(num_edges);
  if (cap_multi > 0) {
    const unsigned nf = (unsigned)ceil_div(cap_multi * 32, 256);
    if (vec) {
      mean_agg_finalize_kernel<true><<<nf, 256, 0, stream>>>(cap_multi, F, indptr, p.header, p.multi, partial, out);
    } else {
      mean_agg_finalize_kernel<false><<<nf, 256, 0, stream>>>(cap_multi, F, indptr, p.header, p.multi, partial, out);
    }
    TTG_LAUNCH_CHECK();
  }
  return TTG_OK;
}

extern "C" int ttg_spmm_csr_fwd(int64_t num_dst, int32_t F, const int64_t* indptr,
                                const int32_t* indices, const float* edge_weight, int32_t mean,
                                const float* x, float* out, void* stream) {
  TTG_CHECK_ARG(F > 0, "spmm_csr_fwd: F=%d must be positive", F);
  if (num_dst == 0) return TTG_OK;
  TTG_CHECK_ARG(indptr && out, "spmm_csr_fwd: null pointer");
  if (F % 4 != 0) {
    spmm_fwd_scalar_kernel<<<(unsigned)ceil_div(num_dst * 32, 256), 256, 0, (cudaStream_t)stream>>>(
        num_dst, F, indptr, indices, edge_weight, mean, x, out);
    TTG_LAUNCH_CHECK();
    return TTG_OK;
  }
  spmm_fwd_kernel<<<(unsigned)ceil_div(num_dst * 32, 256), 256, 0, (cudaStream_t)stream>>>(
      num_dst, F, indptr, indices, edge_weight, mean, x, out);
  TTG_LAUNCH_CHECK();
  return TTG_OK;
}

extern "C" int ttg_spmm_csr_bwd(int64_t num_dst, int32_t F, const int64_t* indptr,
                                const int32_t* indices, const float* edge_weight, int32_t mean,
                                const float* dout, float* dx, void* stream) {
  TTG_CHECK_ARG(F > 0, "spmm_csr_bwd: F=%d must be positive", F);
  if (num_dst == 0) return TTG_OK;
  TTG_CHECK_ARG(indptr && dout && dx, "spmm_csr_bwd: null pointer");
  if (F % 4 != 0) {
    spmm_bwd_scalar_kernel<<<(unsigned)ceil_div(num_dst * 32, 256), 256, 0, (cudaStream_t)stream>>>(
        num_dst, F, indptr, indices, edge_weight, mean, dout, dx);
    TTG_LAUNCH_CHECK();
    return TTG_OK;
  }
  spmm_bwd_kernel<<<(unsigned)ceil_div(num_dst * 32, 256), 256, 0, (cudaStream_t)stream>>>(
      num_dst, F, indptr, indices, edge_weight, mean, dout, dx);
  TTG_LAUNCH_CHECK();
  return TTG_OK;
}
