// graph.cuh -- CSR pieces shared by the device reordering code (rcm.cu, kway.cu, reorder.cu).
#pragma once

#include "common.cuh"

namespace ttg {

constexpr int64_t kMaxNodes = INT32_MAX;           // rcm, permute: node ids are int32, 1 <= n < 2^31
constexpr int64_t kKwayMaxNodes = INT32_MAX - 1;   // kway: the bound of its host step, ttg_partition_kway_initial
constexpr int64_t kMaxEdges = (int64_t)1 << 40;    // keeps 2 * nnz sort items and their workspaces far from overflow

inline bool nodes_in_range(int64_t n, int64_t max_nodes = kMaxNodes) { return n > 0 && n <= max_nodes; }
inline bool edges_in_range(int64_t nnz) { return nnz >= 0 && nnz <= kMaxEdges; }

// the caller's workspace holds the `need` bytes its sizes carve
inline int check_workspace(const char* who, const void* ws, size_t bytes, size_t need) {
  if (ws && bytes >= need) return TTG_OK;
  set_error("%s: workspace %zu bytes, need %zu", who, bytes, need);
  return TTG_ENOMEM;
}

// blocks of `block` threads covering `threads` threads, at least one
inline unsigned grid(int64_t threads, int block = 256) { return (unsigned)ceil_div(threads > 0 ? threads : 1, block); }

namespace {

// row v of an indptr of n rows over nnz entries is well formed: 0 <= lo <= hi <= nnz, the first row starts at 0 and
// the last one ends at nnz.  When every row passes, indptr is a CSR of exactly nnz entries.
__device__ __forceinline__ bool csr_row(const int64_t* __restrict__ indptr, int64_t n, int64_t nnz, int64_t v,
                                        int64_t* lo, int64_t* hi) {
  *lo = __ldg(indptr + v);
  *hi = __ldg(indptr + v + 1);
  return *lo >= 0 && *lo <= *hi && *hi <= nnz && (v > 0 || *lo == 0) && (v < n - 1 || *hi == nnz);
}

__device__ __forceinline__ int64_t lower_bound_u64(const uint64_t* a, int64_t len, uint64_t x) {
  int64_t lo = 0, hi = len;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (a[mid] < x) lo = mid + 1;
    else hi = mid;
  }
  return lo;
}

// the column of each of the *count sorted (row << colbits | col) keys
__global__ void __launch_bounds__(256)
key_cols_kernel(const int64_t* __restrict__ count, uint64_t colmask, const uint64_t* __restrict__ keys,
                int32_t* __restrict__ cols) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < *count) cols[i] = (int32_t)(keys[i] & colmask);
}

}  // namespace
}  // namespace ttg
