// kway.cu -- multilevel k-way graph partitioner on the DEVICE (SURVEY 8f-3), the scheme of kway_host.cu with
// every data-parallel step on the GPU.  Python (reorder.kway_partition_device) drives it level by level:
//
//   ttg_kway_symmetrise  the in-neighbour CSR becomes the undirected weighted graph kway_host.cu builds:
//                        (v, u) and (u, v) for every edge with u != v, radix sort of the 64-bit keys, run-length
//                        reduction (weight = number of directed edges between the pair), unit vertex weights;
//   ttg_kway_coarsen     one level: handshake heavy-edge matching (every unmatched vertex proposes its heaviest
//                        unmatched neighbour within the vertex-weight bound, ties on a hash of (seed, pair);
//                        mutual proposals match; kMatchRounds rounds), a two-hop pass (unmatched vertices of
//                        degree <= 8 sharing a heaviest neighbour, and isolated vertices, paired through a sort),
//                        coarse ids from a scan over the match leaders, contraction by a sort of the
//                        (cmap[v], cmap[u]) keys and a reduction of their weights; one read-back per level (the
//                        coarse vertex and edge counts);
//   (host step)          the coarsest graph goes to the host, where kway_host.cu's eight grown trials with their
//                        refinement give the initial parts (ttg_partition_kway_initial);
//   ttg_kway_refine      projection onto the next finer level, then synchronous label propagation in the manner
//                        of Jet (Gilbert et al. 2023): every vertex's connectivity to its adjacent parts, the best
//                        target with positive gain, an afterburner that recomputes each candidate's gain as if
//                        its higher-priority neighbours had moved already and drops those no longer positive,
//                        admission into every destination (and out of every source) in priority order by a sort
//                        and a prefix sum of vertex weights against the bounds; a rebalancing step (moves to
//                        adjacent parts first, then an exact fill of the remaining quotas) whenever a part is out
//                        of its bounds.  The bounds are the host's, 1.3 x wider on every level but the finest;
//                        on the finest level (unit weights) the call guarantees the exact bound;
//   ttg_kway_edge_cut    input edges whose ends lie in different parts.
//
// Determinism: the labels depend on the graph and the seed alone.  Decisions use integer arithmetic, stable
// radix sorts and hashed tie-breaks; the atomics that remain are integer sums (order-free) and hash-table
// inserts whose final contents do not depend on the order they land in.
//
// The result meets the host partitioner's balance bounds and its cut quality on the tested graphs; it is NOT the
// host partitioner's partition (different matching and refinement), and not METIS' either.
#include <algorithm>
#include <vector>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_select.cuh>
#include <thrust/iterator/counting_iterator.h>

#include "common.cuh"

namespace ttg {
namespace {

constexpr int kMatchRounds = 8;
constexpr int64_t kSmallDegree = 8;          // two-hop pass: the host's bound
constexpr int kLightDegree = 512;            // up to here a warp holds the vertex's part table in shared memory
constexpr int kWarpTable = 2 * kLightDegree; // slots per warp (load factor <= 1/2)
constexpr int kWarpsPerBlock = 4;
constexpr int kHeavyThreads = 256;
constexpr int kHeavyRange = 8192;            // part ids per pass of a heavy vertex's direct-indexed table
constexpr int kItersPerPass = 3;             // label-propagation iterations per refine pass
constexpr int kLocalRebalanceRounds = 6;
constexpr int64_t kInf = INT64_MAX / 4;

enum Mode { M_REFINE = 0, M_REBALANCE = 1, M_FILL = 2 };

__host__ __device__ __forceinline__ uint64_t mix64(uint64_t z) {
  z += 0x9e3779b97f4a7c15ull;
  z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
  z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
  return z ^ (z >> 31);
}
__device__ __forceinline__ uint32_t hash32(uint64_t salt, uint64_t x) { return (uint32_t)(mix64(salt ^ mix64(x)) >> 32); }

// higher = moves first: the gain, then a hash of (salt, v)
__device__ __forceinline__ uint64_t move_prio(int32_t gain, int32_t v, uint64_t salt) {
  return ((uint64_t)((uint32_t)gain ^ 0x80000000u) << 32) | hash32(salt, (uint64_t)v);
}

__device__ __forceinline__ uint64_t warp_max_u64(uint64_t x) {
  for (int o = 16; o > 0; o >>= 1) {
    const uint64_t y = __shfl_xor_sync(0xffffffffu, x, o);
    x = y > x ? y : x;
  }
  return x;
}
__device__ __forceinline__ int64_t warp_sum_i64(int64_t x) {
  for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
  return x;
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

// ---- sorted (row, col) keys -> weighted CSR -----------------------------------------------------------------
// keys are (row << colbits) | col, sorted, with the dropped entries (self pairs, keyed `drop`) last.  The first
// entry of every run of equal keys is its head; pos = exclusive scan of the heads gives each run its slot.
__global__ void __launch_bounds__(256)
run_heads_kernel(int64_t items, uint64_t drop, const uint64_t* __restrict__ keys, int64_t* __restrict__ pos) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= items) return;
  const uint64_t k = keys[i];
  pos[i] = (k != drop && (i == 0 || keys[i - 1] != k)) ? 1 : 0;
}

// after the scan: the run's key and summed weight in its slot (weights == nullptr: 1 per entry); counts[1] = runs
__global__ void __launch_bounds__(256)
run_reduce_kernel(int64_t items, uint64_t drop, const uint64_t* __restrict__ keys, const int64_t* __restrict__ pos,
                  const int32_t* __restrict__ weights, uint64_t* __restrict__ ukeys, int32_t* __restrict__ uw,
                  int64_t* __restrict__ counts) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= items) return;
  const uint64_t k = keys[i];
  const bool head = k != drop && (i == 0 || keys[i - 1] != k);
  if (i == items - 1) counts[1] = pos[i] + (head ? 1 : 0);
  if (k == drop) return;
  const int64_t slot = pos[i] + (head ? 0 : -1);
  if (head) ukeys[slot] = k;
  atomicAdd(uw + slot, weights ? weights[i] : 1);
}

// row r's bounds by binary search over the m distinct keys; the column of every entry; rows > counts[0] idle
__global__ void __launch_bounds__(256)
csr_rows_kernel(int64_t max_rows, const int64_t* __restrict__ counts, int colbits, const uint64_t* __restrict__ ukeys,
                int64_t* __restrict__ xadj) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t rows = counts[0], m = counts[1];
  if (r > rows || r > max_rows) return;
  xadj[r] = r == rows ? m : lower_bound_u64(ukeys, m, (uint64_t)r << colbits);
}

__global__ void __launch_bounds__(256)
csr_cols_kernel(const int64_t* __restrict__ counts, uint64_t colmask, const uint64_t* __restrict__ ukeys,
                int32_t* __restrict__ adj) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < counts[1]) adj[i] = (int32_t)(ukeys[i] & colmask);
}

// ---- symmetrise ------------------------------------------------------------------------------------------------
// one warp per row v: (v, u) at e and (u, v) at nnz + e, self loops dropped; flags: id out of range / not a CSR
__global__ void __launch_bounds__(256)
sym_emit_kernel(int64_t n, int64_t nnz, int colbits, uint64_t drop, const int64_t* __restrict__ indptr,
                const int32_t* __restrict__ indices, uint64_t* __restrict__ keys, int32_t* __restrict__ flags) {
  const int64_t v = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (v >= n) return;
  const int64_t lo = __ldg(indptr + v), hi = __ldg(indptr + v + 1);
  if (lo < 0 || hi < lo || hi > nnz || (v == 0 && lo != 0) || (v == n - 1 && hi != nnz)) {
    flags[0] = 1;
    return;
  }
  for (int64_t e = lo + lane; e < hi; e += 32) {
    const int32_t u = __ldg(indices + e);
    if (u < 0 || u >= n) flags[0] = 1;
    const bool keep = u >= 0 && u < n && u != v;
    keys[e] = keep ? ((uint64_t)v << colbits) | (uint64_t)u : drop;
    keys[nnz + e] = keep ? ((uint64_t)u << colbits) | (uint64_t)v : drop;
  }
}

__global__ void __launch_bounds__(256)
fill_i32_kernel(int64_t n, int32_t value, int32_t* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = value;
}

// ---- matching ------------------------------------------------------------------------------------------------
// one warp per unmatched vertex: its heaviest unmatched neighbour within the weight bound
__global__ void __launch_bounds__(256)
match_propose_kernel(int64_t n, const int64_t* __restrict__ xadj, const int32_t* __restrict__ adj,
                     const int32_t* __restrict__ adjw, const int32_t* __restrict__ vw, int32_t maxvw,
                     const int32_t* __restrict__ match, int32_t* __restrict__ prop, uint64_t salt) {
  const int64_t v = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (v >= n) return;
  if (match[v] >= 0) {
    if (lane == 0) prop[v] = -1;
    return;
  }
  const int32_t wv = vw[v];
  uint64_t best = 0;
  for (int64_t e = xadj[v] + lane; e < xadj[v + 1]; e += 32) {
    const int32_t u = adj[e];
    if (match[u] >= 0 || wv + vw[u] > maxvw) continue;
    const uint64_t lo = (uint64_t)min((int64_t)u, v), hi = (uint64_t)max((int64_t)u, v);
    const uint64_t key = ((uint64_t)adjw[e] << 32) | hash32(salt, (hi << 32) | lo);
    if (key > best) best = key;
  }
  best = warp_max_u64(best);
  // the key names the pair only up to its hash: find the neighbour that produced it (smallest id on a clash)
  int32_t pick = INT32_MAX;
  if (best != 0)
    for (int64_t e = xadj[v] + lane; e < xadj[v + 1]; e += 32) {
      const int32_t u = adj[e];
      if (match[u] >= 0 || wv + vw[u] > maxvw) continue;
      const uint64_t lo = (uint64_t)min((int64_t)u, v), hi = (uint64_t)max((int64_t)u, v);
      if ((((uint64_t)adjw[e] << 32) | hash32(salt, (hi << 32) | lo)) == best) pick = min(pick, u);
    }
  for (int o = 16; o > 0; o >>= 1) pick = min(pick, __shfl_xor_sync(0xffffffffu, pick, o));
  if (lane == 0) prop[v] = best != 0 ? pick : -1;
}

__global__ void __launch_bounds__(256)
match_accept_kernel(int64_t n, const int32_t* __restrict__ prop, int32_t* __restrict__ match) {
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= n) return;
  const int32_t u = prop[v];
  if (u >= 0 && prop[u] == (int32_t)v) match[v] = u;
}

// two-hop key of every unmatched vertex of degree <= kSmallDegree: (heaviest neighbour, v); isolated vertices
// share the neighbour id n; everything else sorts last
__global__ void __launch_bounds__(256)
twohop_key_kernel(int64_t n, const int64_t* __restrict__ xadj, const int32_t* __restrict__ adj,
                  const int32_t* __restrict__ adjw, const int32_t* __restrict__ match, uint64_t* __restrict__ keys) {
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= n) return;
  const int64_t lo = xadj[v], hi = xadj[v + 1];
  uint64_t key = ~0ull;
  if (match[v] < 0 && hi - lo <= kSmallDegree) {
    int32_t best = (int32_t)n, bw = 0;
    for (int64_t e = lo; e < hi; ++e)
      if (adjw[e] > bw || (adjw[e] == bw && adj[e] < best)) {
        bw = adjw[e];
        best = adj[e];
      }
    key = ((uint64_t)best << 32) | (uint64_t)v;
  }
  keys[v] = key;
}

// sorted two-hop keys: the first of every run of one neighbour, as a running max of run starts
__global__ void __launch_bounds__(256)
twohop_start_kernel(int64_t n, const uint64_t* __restrict__ keys, int32_t* __restrict__ start) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  start[i] = (i == 0 || (keys[i] >> 32) != (keys[i - 1] >> 32)) ? (int32_t)i : 0;
}

// pairs (start, start + 1), (start + 2, start + 3), ... inside every run
__global__ void __launch_bounds__(256)
twohop_pair_kernel(int64_t n, const uint64_t* __restrict__ keys, const int32_t* __restrict__ start,
                   const int32_t* __restrict__ vw, int32_t maxvw, int32_t* __restrict__ match) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i + 1 >= n) return;
  const uint64_t a = keys[i], b = keys[i + 1];
  if (a == ~0ull || b == ~0ull || (a >> 32) != (b >> 32) || ((i - start[i]) & 1)) return;
  const int32_t va = (int32_t)(a & 0xffffffffu), vb = (int32_t)(b & 0xffffffffu);
  if (vw[va] + vw[vb] > maxvw) return;
  match[va] = vb;
  match[vb] = va;
}

// a leader is unmatched or the smaller id of its pair
__global__ void __launch_bounds__(256)
leader_kernel(int64_t n, const int32_t* __restrict__ match, int32_t* __restrict__ lead) {
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v < n) lead[v] = (match[v] < 0 || (int32_t)v < match[v]) ? 1 : 0;
}

// cmap of both members, coarse vertex weights, counts[0] = coarse vertices
__global__ void __launch_bounds__(256)
cmap_kernel(int64_t n, const int32_t* __restrict__ match, const int32_t* __restrict__ lead,
            const int32_t* __restrict__ id, const int32_t* __restrict__ vw, int32_t* __restrict__ cmap,
            int32_t* __restrict__ cvw, int64_t* __restrict__ counts) {
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= n) return;
  if (v == n - 1) counts[0] = (int64_t)id[v] + lead[v];
  if (!lead[v]) return;
  const int32_t c = id[v], u = match[v];
  cmap[v] = c;
  if (u >= 0) cmap[u] = c;
  cvw[c] = vw[v] + (u >= 0 ? vw[u] : 0);
}

// one warp per fine vertex: (cmap[v], cmap[u]) with the edge weight; pairs inside one coarse vertex dropped
__global__ void __launch_bounds__(256)
contract_emit_kernel(int64_t n, int colbits, uint64_t drop, const int64_t* __restrict__ xadj,
                     const int32_t* __restrict__ adj, const int32_t* __restrict__ adjw,
                     const int32_t* __restrict__ cmap, uint64_t* __restrict__ keys, int32_t* __restrict__ w) {
  const int64_t v = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (v >= n) return;
  const uint64_t cv = (uint64_t)cmap[v];
  for (int64_t e = xadj[v] + lane; e < xadj[v + 1]; e += 32) {
    const uint64_t cu = (uint64_t)cmap[adj[e]];
    keys[e] = cu == cv ? drop : (cv << colbits) | cu;
    w[e] = adjw[e];
  }
}

// ---- refinement ---------------------------------------------------------------------------------------------
struct Bounds {
  int64_t maxpw, minpw;
};

// may v (weight wv, part a) go to q?  refine: any adjacent part with room; rebalance: from an overweight part to
// any adjacent part with room, else only into an underweight part
__device__ __forceinline__ bool eligible(int mode, int32_t q, int32_t a, int32_t wv, const int64_t* pw, Bounds b) {
  if (q == a || pw[q] + wv > b.maxpw) return false;
  return mode == M_REFINE || pw[a] > b.maxpw || pw[q] < b.minpw;
}

// the outcome of a vertex's scan: dest = -1 (stays) or the target, its gain, and the candidate flag
__device__ __forceinline__ void settle(int mode, int32_t v, int32_t a, int32_t wv, int64_t own, uint64_t best,
                                      const int64_t* pw, Bounds b, int32_t* dest, int32_t* gain, uint8_t* cand) {
  int32_t d = -1, g = 0;
  if (best != 0) {
    d = (int32_t)(best & 0xffffffffu);
    g = (int32_t)((int64_t)(best >> 32) - 1 - own);
  }
  bool ok = d >= 0;
  if (mode == M_REFINE) ok = ok && g > 0 && pw[a] - wv >= b.minpw;
  else ok = ok && (pw[a] > b.maxpw || pw[a] - wv >= b.minpw);
  dest[v] = ok ? d : -1;
  gain[v] = g;
  cand[v] = ok ? 1 : 0;
}

// one warp per vertex of degree <= kLightDegree: connectivity to every adjacent part in a shared-memory hash table
// (the final contents do not depend on the order of the inserts), then the best eligible part:
// max (connection, hash(salt, v, part)); best packs (connection + 1) << 32 | part
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
move_light_kernel(int mode, int64_t n, const int64_t* __restrict__ xadj, const int32_t* __restrict__ adj,
                  const int32_t* __restrict__ adjw, const int32_t* __restrict__ vw, const int32_t* __restrict__ part,
                  const int64_t* __restrict__ pw, Bounds b, uint64_t salt, int32_t* __restrict__ dest,
                  int32_t* __restrict__ gain, uint8_t* __restrict__ cand) {
  __shared__ int32_t tkey[kWarpsPerBlock][kWarpTable];
  __shared__ int32_t tval[kWarpsPerBlock][kWarpTable];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t v = (int64_t)blockIdx.x * kWarpsPerBlock + warp;
  if (v >= n) return;
  const int64_t lo = xadj[v], hi = xadj[v + 1];
  if (hi - lo > kLightDegree) return;   // move_heavy_kernel
  int size = 32;
  while (size < 2 * (hi - lo)) size <<= 1;
  int32_t* keys = tkey[warp];
  int32_t* vals = tval[warp];
  for (int i = lane; i < size; i += 32) {
    keys[i] = -1;
    vals[i] = 0;
  }
  __syncwarp();
  const int32_t a = part[v], wv = vw[v];
  int64_t own = 0;
  for (int64_t e = lo + lane; e < hi; e += 32) {
    const int32_t p = part[adj[e]], w = adjw[e];
    if (p == a) {
      own += w;
      continue;
    }
    uint32_t h = ((uint32_t)p * 0x9e3779b1u) >> 7;
    for (;;) {
      h &= (uint32_t)(size - 1);
      const int32_t k = atomicCAS(keys + h, -1, p);
      if (k == -1 || k == p) {
        atomicAdd(vals + h, w);
        break;
      }
      ++h;
    }
  }
  __syncwarp();
  own = warp_sum_i64(own);
  uint64_t best = 0;
  for (int i = lane; i < size; i += 32) {
    const int32_t q = keys[i];
    if (q < 0 || !eligible(mode, q, a, wv, pw, b)) continue;
    // the table is ordered by connection; among equal connections by a hash of (v, part)
    const uint64_t key = ((uint64_t)(vals[i] + 1) << 32) | hash32(salt ^ (uint64_t)v, (uint64_t)q);
    if (key > best) best = key;
  }
  best = warp_max_u64(best);
  int32_t pick = -1;   // the part behind the winning key
  for (int i = lane; i < size; i += 32) {
    const int32_t q = keys[i];
    if (best != 0 && q >= 0 && ((uint64_t)(vals[i] + 1) << 32 | hash32(salt ^ (uint64_t)v, (uint64_t)q)) == best &&
        eligible(mode, q, a, wv, pw, b))
      pick = max(pick, q);
  }
  for (int o = 16; o > 0; o >>= 1) pick = max(pick, __shfl_xor_sync(0xffffffffu, pick, o));
  if (lane == 0)
    settle(mode, (int32_t)v, a, wv, own, best ? ((best >> 32) << 32) | (uint32_t)pick : 0, pw, b, dest, gain, cand);
}

// one block per vertex of degree > kLightDegree: connections in a direct-indexed shared table, kHeavyRange part
// ids per pass over the neighbours
__global__ void __launch_bounds__(kHeavyThreads)
move_heavy_kernel(int mode, int64_t n, int32_t k, const int32_t* __restrict__ heavy, const int64_t* __restrict__ xadj,
                  const int32_t* __restrict__ adj, const int32_t* __restrict__ adjw, const int32_t* __restrict__ vw,
                  const int32_t* __restrict__ part, const int64_t* __restrict__ pw, Bounds b, uint64_t salt,
                  int32_t* __restrict__ dest, int32_t* __restrict__ gain, uint8_t* __restrict__ cand) {
  __shared__ int32_t conn[kHeavyRange];
  __shared__ uint64_t red_best[kHeavyThreads / 32];
  __shared__ int64_t red_own[kHeavyThreads / 32];
  const int32_t v = heavy[blockIdx.x];
  const int64_t lo = xadj[v], hi = xadj[v + 1];
  const int32_t a = part[v], wv = vw[v];
  uint64_t best = 0;   // (connection + 1) << 32 | part, after the hash order below
  uint32_t best_hash = 0;
  int64_t own = 0;
  for (int32_t r0 = 0; r0 < k; r0 += kHeavyRange) {
    for (int i = threadIdx.x; i < kHeavyRange; i += kHeavyThreads) conn[i] = 0;
    __syncthreads();
    for (int64_t e = lo + threadIdx.x; e < hi; e += kHeavyThreads) {
      const int32_t p = part[adj[e]];
      if (r0 == 0 && p == a) own += adjw[e];
      if (p != a && p >= r0 && p < r0 + kHeavyRange) atomicAdd(conn + (p - r0), adjw[e]);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < kHeavyRange && r0 + i < k; i += kHeavyThreads) {
      const int32_t q = r0 + i;
      if (conn[i] == 0 || !eligible(mode, q, a, wv, pw, b)) continue;
      const uint32_t h = hash32(salt ^ (uint64_t)v, (uint64_t)q);
      const uint64_t c = (uint64_t)(conn[i] + 1);
      if (c > (best >> 32) || (c == (best >> 32) && (h > best_hash || (h == best_hash && (uint32_t)q > (uint32_t)best)))) {
        best = (c << 32) | (uint32_t)q;
        best_hash = h;
      }
    }
    __syncthreads();
  }
  // block max of (connection, hash, part) and sum of own
  uint64_t key_hi = best >> 32, key_lo = ((uint64_t)best_hash << 32) | (best & 0xffffffffu);
  own = warp_sum_i64(own);
  for (int o = 16; o > 0; o >>= 1) {
    const uint64_t oh = __shfl_xor_sync(0xffffffffu, key_hi, o), ol = __shfl_xor_sync(0xffffffffu, key_lo, o);
    if (oh > key_hi || (oh == key_hi && ol > key_lo)) {
      key_hi = oh;
      key_lo = ol;
    }
  }
  __shared__ uint64_t red_lo[kHeavyThreads / 32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) {
    red_best[warp] = key_hi;
    red_lo[warp] = key_lo;
    red_own[warp] = own;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    uint64_t bh = 0, bl = 0;
    int64_t o = 0;
    for (int w = 0; w < kHeavyThreads / 32; ++w) {
      o += red_own[w];
      if (red_best[w] > bh || (red_best[w] == bh && red_lo[w] > bl)) {
        bh = red_best[w];
        bl = red_lo[w];
      }
    }
    settle(mode, v, a, wv, o, bh ? (bh << 32) | (bl & 0xffffffffu) : 0, pw, b, dest, gain, cand);
  }
}

__global__ void __launch_bounds__(256)
heavy_list_kernel(int64_t n, const int64_t* __restrict__ xadj, int32_t* __restrict__ heavy, int32_t* __restrict__ count) {
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  // the list's order varies from run to run; every entry's result lands at its own vertex
  if (v < n && xadj[v + 1] - xadj[v] > kLightDegree) heavy[atomicAdd(count, 1)] = (int32_t)v;
}

// one warp per candidate: its gain if every neighbour of higher priority had moved already; kept if positive
__global__ void __launch_bounds__(256)
afterburn_kernel(int64_t n, const int64_t* __restrict__ xadj, const int32_t* __restrict__ adj,
                 const int32_t* __restrict__ adjw, const int32_t* __restrict__ part, const int32_t* __restrict__ dest,
                 const int32_t* __restrict__ gain, uint64_t salt, uint8_t* __restrict__ cand) {
  const int64_t v = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (v >= n || dest[v] < 0) return;
  const int32_t a = part[v], d = dest[v];
  const uint64_t pv = move_prio(gain[v], (int32_t)v, salt);
  int64_t g = 0;
  for (int64_t e = xadj[v] + lane; e < xadj[v + 1]; e += 32) {
    const int32_t u = adj[e];
    int32_t pu = part[u];
    const int32_t du = dest[u];
    if (du >= 0 && move_prio(gain[u], u, salt) > pv) pu = du;
    g += pu == d ? adjw[e] : (pu == a ? -adjw[e] : 0);
  }
  g = warp_sum_i64(g);
  if (lane == 0) cand[v] = g > 0 ? 1 : 0;
}

// sort key of every listed vertex: moves by descending priority; fill leavers by ascending internal connection
__global__ void __launch_bounds__(256)
prio_key_kernel(int64_t c, int mode, const int32_t* __restrict__ list, const int32_t* __restrict__ gain,
                const int64_t* __restrict__ internal, uint64_t salt, uint64_t* __restrict__ keys,
                int32_t* __restrict__ vals) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= c) return;
  const int32_t v = list[i];
  keys[i] = mode == M_FILL ? ((uint64_t)internal[v] << 32) | hash32(salt, (uint64_t)v)
                           : ~move_prio(gain[v], v, salt);
  vals[i] = v;
}

__global__ void __launch_bounds__(256)
part_key_kernel(int64_t c, const int32_t* __restrict__ order, const int32_t* __restrict__ of,
                uint32_t* __restrict__ keys, int32_t* __restrict__ vals) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= c) return;
  const int32_t v = order[i];
  keys[i] = (uint32_t)of[v];
  vals[i] = v;
}

__global__ void __launch_bounds__(256)
weights_kernel(int64_t c, const int32_t* __restrict__ vals, const int32_t* __restrict__ vw, int64_t* __restrict__ w) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < c) w[i] = vw[vals[i]];
}

__global__ void __launch_bounds__(256)
seg_start_kernel(int64_t c, const uint32_t* __restrict__ keys, int32_t* __restrict__ start) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < c && (i == 0 || keys[i] != keys[i - 1])) start[keys[i]] = (int32_t)i;
}

// inside each part's segment (priority order): admitted while the inclusive weight stays within hi[part] and
// the weight before it is below cover[part]
__global__ void __launch_bounds__(256)
admit_kernel(int64_t c, const uint32_t* __restrict__ keys, const int32_t* __restrict__ vals,
             const int64_t* __restrict__ excl, const int32_t* __restrict__ vw, const int32_t* __restrict__ start,
             const int64_t* __restrict__ hi, const int64_t* __restrict__ cover, uint8_t* __restrict__ ok) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= c) return;
  const uint32_t p = keys[i];
  const int32_t v = vals[i];
  const int64_t before = excl[i] - excl[start[p]];
  ok[v] = (before + vw[v] <= hi[p] && before < cover[p]) ? 1 : 0;
}

__global__ void __launch_bounds__(256)
apply_kernel(int64_t c, const int32_t* __restrict__ list, const uint8_t* __restrict__ ok_in,
             const uint8_t* __restrict__ ok_out, const int32_t* __restrict__ dest, const int32_t* __restrict__ vw,
             int32_t* __restrict__ part, unsigned long long* __restrict__ pw, unsigned long long* __restrict__ moved) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= c) return;
  const int32_t v = list[i];
  if (!ok_in[v] || !ok_out[v]) return;
  const int32_t from = part[v], to = dest[v];
  part[v] = to;
  atomicAdd(pw + to, (unsigned long long)vw[v]);
  atomicAdd(pw + from, (unsigned long long)(-(int64_t)vw[v]));
  atomicAdd(moved, 1ull);
}

// per-part limits of a round: room (inflow), want (inflow cover), spare (outflow), give (outflow cover)
__global__ void __launch_bounds__(256)
limits_kernel(int32_t k, int mode, const int64_t* __restrict__ pw, Bounds b, int64_t* __restrict__ room,
              int64_t* __restrict__ want, int64_t* __restrict__ spare, int64_t* __restrict__ give) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= k) return;
  const int64_t w = pw[p];
  room[p] = b.maxpw - w;
  want[p] = mode == M_REBALANCE && w < b.minpw ? b.minpw - w : kInf;
  spare[p] = mode == M_FILL ? kInf : w - b.minpw;
  if (mode != M_FILL) give[p] = mode == M_REBALANCE && w > b.maxpw ? w - b.maxpw : kInf;
}

__global__ void __launch_bounds__(256)
part_weights_kernel(int64_t n, const int32_t* __restrict__ part, const int32_t* __restrict__ vw,
                    unsigned long long* __restrict__ pw, int32_t k, int32_t* __restrict__ bad) {
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= n) return;
  const int32_t p = part[v];
  if (p < 0 || p >= k) {
    *bad = 1;
    return;
  }
  atomicAdd(pw + p, (unsigned long long)vw[v]);
}

__global__ void __launch_bounds__(256)
project_kernel(int64_t n, const int32_t* __restrict__ cmap, const int32_t* __restrict__ coarse_part,
               int32_t* __restrict__ part) {
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v < n) part[v] = coarse_part[cmap[v]];
}

// fill: vertices of parts that must give weight, with their internal connection
__global__ void __launch_bounds__(256)
fill_cand_kernel(int64_t n, const int64_t* __restrict__ xadj, const int32_t* __restrict__ adj,
                 const int32_t* __restrict__ adjw, const int32_t* __restrict__ part, const int64_t* __restrict__ give,
                 int64_t* __restrict__ internal, uint8_t* __restrict__ cand) {
  const int64_t v = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (v >= n) return;
  const int32_t a = part[v];
  if (give[a] <= 0) {
    if (lane == 0) cand[v] = 0;
    return;
  }
  int64_t s = 0;
  for (int64_t e = xadj[v] + lane; e < xadj[v + 1]; e += 32) s += part[adj[e]] == a ? adjw[e] : 0;
  s = warp_sum_i64(s);
  if (lane == 0) {
    internal[v] = s;
    cand[v] = 1;
  }
}

// fill: the leavers in order, each at its weight offset in the concatenated quotas (deficits first, then room)
__global__ void __launch_bounds__(256)
fill_dest_kernel(int64_t c, int32_t k, const int32_t* __restrict__ leavers, const int64_t* __restrict__ excl,
                 const int64_t* __restrict__ cum, int32_t* __restrict__ dest, uint8_t* __restrict__ ok) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= c) return;
  const int32_t v = leavers[i];
  const int64_t at = excl[i];
  int64_t lo = 0, hi = 2 * (int64_t)k;   // first slot whose inclusive end exceeds `at`
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (cum[mid] <= at) lo = mid + 1;
    else hi = mid;
  }
  ok[v] = lo < 2 * (int64_t)k;
  dest[v] = lo < 2 * (int64_t)k ? (int32_t)(lo % k) : -1;
}

__global__ void __launch_bounds__(256)
cut_kernel(int64_t n, const int64_t* __restrict__ indptr, const int32_t* __restrict__ indices,
           const int32_t* __restrict__ part, unsigned long long* __restrict__ cut) {
  const int64_t v = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (v >= n) return;
  const int32_t a = part[v];
  int64_t c = 0;
  for (int64_t e = indptr[v] + lane; e < indptr[v + 1]; e += 32) c += part[indices[e]] != a;
  c = warp_sum_i64(c);
  if (lane == 0 && c) atomicAdd(cut, (unsigned long long)c);
}

// ---- workspaces ---------------------------------------------------------------------------------------------
struct SymWs {
  uint64_t *keys_a, *keys_b;
  int64_t* pos;
  int64_t* counts;   // [0] rows, [1] distinct pairs
  int32_t* flags;
  void* cub_tmp;
  size_t cub_bytes, total;
};

SymWs carve_sym(void* ws, int64_t n, int64_t nnz) {
  SymWs w;
  Carver c{ws};
  const int64_t items = 2 * nnz > 0 ? 2 * nnz : 1;
  w.keys_a = (uint64_t*)c.take(sizeof(uint64_t) * (size_t)items);
  w.keys_b = (uint64_t*)c.take(sizeof(uint64_t) * (size_t)items);
  w.pos = (int64_t*)c.take(sizeof(int64_t) * (size_t)items);
  w.counts = (int64_t*)c.take(sizeof(int64_t) * 2);
  w.flags = (int32_t*)c.take(sizeof(int32_t));
  size_t sort_bytes = 0, scan_bytes = 0;
  cub::DoubleBuffer<uint64_t> dk(nullptr, nullptr);
  cub::DeviceRadixSort::SortKeys(nullptr, sort_bytes, dk, items);
  cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, (int64_t*)nullptr, items);
  w.cub_bytes = std::max(sort_bytes, scan_bytes);
  w.cub_tmp = c.take(w.cub_bytes);
  w.total = c.off;
  return w;
}

struct CoarsenWs {
  int32_t *match, *prop, *lead, *id, *start;
  uint64_t *hkeys_a, *hkeys_b;   // two-hop keys [n]
  uint64_t *keys_a, *keys_b;     // contraction keys [m]
  int32_t *w_a, *w_b;            // contraction weights [m]
  int64_t* pos;                  // [m]
  int64_t* counts;               // [0] coarse vertices, [1] coarse edges
  void* cub_tmp;
  size_t cub_bytes, total;
};

CoarsenWs carve_coarsen(void* ws, int64_t n, int64_t m) {
  CoarsenWs w;
  Carver c{ws};
  const size_t un = (size_t)n, um = (size_t)(m > 0 ? m : 1);
  w.match = (int32_t*)c.take(sizeof(int32_t) * un);
  w.prop = (int32_t*)c.take(sizeof(int32_t) * un);
  w.lead = (int32_t*)c.take(sizeof(int32_t) * un);
  w.id = (int32_t*)c.take(sizeof(int32_t) * un);
  w.start = (int32_t*)c.take(sizeof(int32_t) * un);
  w.hkeys_a = (uint64_t*)c.take(sizeof(uint64_t) * un);
  w.hkeys_b = (uint64_t*)c.take(sizeof(uint64_t) * un);
  w.keys_a = (uint64_t*)c.take(sizeof(uint64_t) * um);
  w.keys_b = (uint64_t*)c.take(sizeof(uint64_t) * um);
  w.w_a = (int32_t*)c.take(sizeof(int32_t) * um);
  w.w_b = (int32_t*)c.take(sizeof(int32_t) * um);
  w.pos = (int64_t*)c.take(sizeof(int64_t) * um);
  w.counts = (int64_t*)c.take(sizeof(int64_t) * 2);
  size_t b1 = 0, b2 = 0, b3 = 0, b4 = 0, b5 = 0;
  cub::DoubleBuffer<uint64_t> dk(nullptr, nullptr);
  cub::DoubleBuffer<int32_t> dv(nullptr, nullptr);
  cub::DeviceRadixSort::SortKeys(nullptr, b1, dk, n);
  cub::DeviceRadixSort::SortPairs(nullptr, b2, dk, dv, (int64_t)um);
  cub::DeviceScan::ExclusiveSum(nullptr, b3, (int32_t*)nullptr, (int32_t*)nullptr, n);
  cub::DeviceScan::InclusiveScan(nullptr, b4, (int32_t*)nullptr, (int32_t*)nullptr, cub::Max(), n);
  cub::DeviceScan::ExclusiveSum(nullptr, b5, (int64_t*)nullptr, (int64_t)um);
  w.cub_bytes = std::max({b1, b2, b3, b4, b5});
  w.cub_tmp = c.take(w.cub_bytes);
  w.total = c.off;
  return w;
}

struct RefineWs {
  int64_t *pw, *room, *want, *spare, *give, *cum;   // [k] x 5, cum [2k]
  int32_t* start;                                    // [k]
  int32_t *dest, *gain, *list, *order, *heavy;       // [n]
  int64_t *internal, *excl;                          // [n]
  uint64_t *keys_a, *keys_b;                         // [n]
  uint32_t *pkeys_a, *pkeys_b;                       // [n]
  int32_t *vals_a, *vals_b;                          // [n]
  uint8_t *cand, *ok_in, *ok_out;                    // [n]
  int32_t* counts;                                   // [0] selected, [1] heavy, [2] bad part id
  unsigned long long* moved;
  void* cub_tmp;
  size_t cub_bytes, total;
};

RefineWs carve_refine(void* ws, int64_t n, int32_t k) {
  RefineWs w;
  Carver c{ws};
  const size_t un = (size_t)n, uk = (size_t)k;
  w.pw = (int64_t*)c.take(sizeof(int64_t) * uk);
  w.room = (int64_t*)c.take(sizeof(int64_t) * uk);
  w.want = (int64_t*)c.take(sizeof(int64_t) * uk);
  w.spare = (int64_t*)c.take(sizeof(int64_t) * uk);
  w.give = (int64_t*)c.take(sizeof(int64_t) * uk);
  w.cum = (int64_t*)c.take(sizeof(int64_t) * 2 * uk);
  w.start = (int32_t*)c.take(sizeof(int32_t) * uk);
  w.dest = (int32_t*)c.take(sizeof(int32_t) * un);
  w.gain = (int32_t*)c.take(sizeof(int32_t) * un);
  w.list = (int32_t*)c.take(sizeof(int32_t) * un);
  w.order = (int32_t*)c.take(sizeof(int32_t) * un);
  w.heavy = (int32_t*)c.take(sizeof(int32_t) * un);
  w.internal = (int64_t*)c.take(sizeof(int64_t) * un);
  w.excl = (int64_t*)c.take(sizeof(int64_t) * un);
  w.keys_a = (uint64_t*)c.take(sizeof(uint64_t) * un);
  w.keys_b = (uint64_t*)c.take(sizeof(uint64_t) * un);
  w.pkeys_a = (uint32_t*)c.take(sizeof(uint32_t) * un);
  w.pkeys_b = (uint32_t*)c.take(sizeof(uint32_t) * un);
  w.vals_a = (int32_t*)c.take(sizeof(int32_t) * un);
  w.vals_b = (int32_t*)c.take(sizeof(int32_t) * un);
  w.cand = (uint8_t*)c.take(un);
  w.ok_in = (uint8_t*)c.take(un);
  w.ok_out = (uint8_t*)c.take(un);
  w.counts = (int32_t*)c.take(sizeof(int32_t) * 4);
  w.moved = (unsigned long long*)c.take(sizeof(unsigned long long));
  size_t b1 = 0, b2 = 0, b3 = 0, b4 = 0;
  cub::DeviceSelect::Flagged(nullptr, b1, thrust::counting_iterator<int32_t>(0), (const uint8_t*)nullptr,
                             (int32_t*)nullptr, (int32_t*)nullptr, n);
  cub::DoubleBuffer<uint64_t> dk(nullptr, nullptr);
  cub::DoubleBuffer<uint32_t> pk(nullptr, nullptr);
  cub::DoubleBuffer<int32_t> dv(nullptr, nullptr);
  cub::DeviceRadixSort::SortPairs(nullptr, b2, dk, dv, n);
  cub::DeviceRadixSort::SortPairs(nullptr, b3, pk, dv, n);
  cub::DeviceScan::ExclusiveSum(nullptr, b4, (int64_t*)nullptr, (int64_t*)nullptr, n);
  w.cub_bytes = std::max({b1, b2, b3, b4});
  w.cub_tmp = c.take(w.cub_bytes);
  w.total = c.off;
  return w;
}

bool nodes_in_range(int64_t n) { return n > 0 && n < ((int64_t)1 << 31) - 1; }
bool edges_in_range(int64_t m) { return m >= 0 && m <= ((int64_t)1 << 40); }
unsigned grid(int64_t threads, int block = 256) { return (unsigned)ceil_div(threads > 0 ? threads : 1, block); }

// sorted (row, col) keys in keys (drop last) -> xadj / adj / adjw; counts[0] must hold the row count
int keys_to_csr(int64_t items, int colbits, uint64_t drop, cub::DoubleBuffer<uint64_t>& dk, const int32_t* weights,
                int64_t max_rows, int64_t* pos, int64_t* counts, void* cub_tmp, size_t cub_bytes, int64_t* xadj,
                int32_t* adj, int32_t* adjw, cudaStream_t stream) {
  uint64_t* ukeys = dk.Alternate();
  run_heads_kernel<<<grid(items), 256, 0, stream>>>(items, drop, dk.Current(), pos);
  TTG_LAUNCH_CHECK();
  size_t bytes = cub_bytes;
  TTG_CUDA(cub::DeviceScan::ExclusiveSum(cub_tmp, bytes, pos, items, stream));
  count_launch();
  TTG_CUDA(cudaMemsetAsync(adjw, 0, sizeof(int32_t) * (size_t)items, stream));
  run_reduce_kernel<<<grid(items), 256, 0, stream>>>(items, drop, dk.Current(), pos, weights, ukeys, adjw, counts);
  TTG_LAUNCH_CHECK();
  csr_rows_kernel<<<grid(max_rows + 1), 256, 0, stream>>>(max_rows, counts, colbits, ukeys, xadj);
  TTG_LAUNCH_CHECK();
  csr_cols_kernel<<<grid(items), 256, 0, stream>>>(counts, (1ull << colbits) - 1, ukeys, adj);
  TTG_LAUNCH_CHECK();
  return TTG_OK;
}

// ---- refinement driver --------------------------------------------------------------------------------------
struct Level {
  int64_t n;
  const int64_t* xadj;
  const int32_t* adj;
  const int32_t* adjw;
  const int32_t* vw;
};

struct Refine {
  Level g;
  int32_t k;
  Bounds b;
  uint64_t seed;
  int32_t* part;
  RefineWs w;
  int32_t heavy = 0;
  int64_t salt_counter = 0;
  cudaStream_t stream;

  uint64_t salt() { return mix64(seed ^ mix64(0x6b776179ull + (uint64_t)(salt_counter++))); }

  int part_weights() {
    TTG_CUDA(cudaMemsetAsync(w.pw, 0, sizeof(int64_t) * (size_t)k, stream));
    part_weights_kernel<<<grid(g.n), 256, 0, stream>>>(g.n, part, g.vw, (unsigned long long*)w.pw, k, w.counts + 2);
    TTG_LAUNCH_CHECK();
    return TTG_OK;
  }

  int moves(int mode, uint64_t s) {
    const int64_t n = g.n;
    move_light_kernel<<<grid(n, kWarpsPerBlock), kWarpsPerBlock * 32, 0, stream>>>(
        mode, n, g.xadj, g.adj, g.adjw, g.vw, part, w.pw, b, s, w.dest, w.gain, w.cand);
    TTG_LAUNCH_CHECK();
    if (heavy > 0) {
      move_heavy_kernel<<<(unsigned)heavy, kHeavyThreads, 0, stream>>>(mode, n, k, w.heavy, g.xadj, g.adj, g.adjw,
                                                                      g.vw, part, w.pw, b, s, w.dest, w.gain, w.cand);
      TTG_LAUNCH_CHECK();
    }
    if (mode == M_REFINE) {
      afterburn_kernel<<<grid(n * 32), 256, 0, stream>>>(n, g.xadj, g.adj, g.adjw, part, w.dest, w.gain, s, w.cand);
      TTG_LAUNCH_CHECK();
    }
    return TTG_OK;
  }

  // the flagged vertices in id order -> w.order sorted by priority; *c = their number
  int collect(int mode, uint64_t s, int64_t* c) {
    size_t bytes = w.cub_bytes;
    TTG_CUDA(cub::DeviceSelect::Flagged(w.cub_tmp, bytes, thrust::counting_iterator<int32_t>(0), w.cand, w.list,
                                        w.counts, g.n, stream));
    count_launch();
    int32_t sel = 0;
    TTG_RC(read_back(&sel, w.counts, stream));
    *c = sel;
    if (sel == 0) return TTG_OK;
    prio_key_kernel<<<grid(sel), 256, 0, stream>>>(sel, mode, w.list, w.gain, w.internal, s, w.keys_a, w.vals_a);
    TTG_LAUNCH_CHECK();
    cub::DoubleBuffer<uint64_t> dk(w.keys_a, w.keys_b);
    cub::DoubleBuffer<int32_t> dv(w.vals_a, w.vals_b);
    bytes = w.cub_bytes;
    TTG_CUDA(cub::DeviceRadixSort::SortPairs(w.cub_tmp, bytes, dk, dv, (int64_t)sel, 0, 64, stream));
    count_launch();
    TTG_CUDA(cudaMemcpyAsync(w.order, dv.Current(), sizeof(int32_t) * (size_t)sel, cudaMemcpyDeviceToDevice, stream));
    return TTG_OK;
  }

  // w.order (priority order) grouped by the part `of[v]`, stably; ok[v] from the part's limits.  The grouped list
  // stays in *sorted_vals, the weight offsets in w.excl
  int admit(int64_t c, const int32_t* of, const int64_t* hi, const int64_t* cover, uint8_t* ok,
            int32_t** sorted_vals) {
    part_key_kernel<<<grid(c), 256, 0, stream>>>(c, w.order, of, w.pkeys_a, w.vals_a);
    TTG_LAUNCH_CHECK();
    cub::DoubleBuffer<uint32_t> dk(w.pkeys_a, w.pkeys_b);
    cub::DoubleBuffer<int32_t> dv(w.vals_a, w.vals_b);
    size_t bytes = w.cub_bytes;
    TTG_CUDA(cub::DeviceRadixSort::SortPairs(w.cub_tmp, bytes, dk, dv, c, 0, std::max(1, bits_for((uint64_t)(k - 1))),
                                             stream));
    count_launch();
    weights_kernel<<<grid(c), 256, 0, stream>>>(c, dv.Current(), g.vw, w.excl);
    TTG_LAUNCH_CHECK();
    bytes = w.cub_bytes;
    TTG_CUDA(cub::DeviceScan::ExclusiveSum(w.cub_tmp, bytes, w.excl, w.excl, c, stream));
    count_launch();
    seg_start_kernel<<<grid(c), 256, 0, stream>>>(c, dk.Current(), w.start);
    TTG_LAUNCH_CHECK();
    admit_kernel<<<grid(c), 256, 0, stream>>>(c, dk.Current(), dv.Current(), w.excl, g.vw, w.start, hi, cover, ok);
    TTG_LAUNCH_CHECK();
    if (sorted_vals) *sorted_vals = dv.Current();
    return TTG_OK;
  }

  // one round of moves in `mode` (refine / local rebalance); *moved = number of vertices that moved
  int round(int mode, int64_t* moved) {
    const uint64_t s = salt();
    TTG_RC(moves(mode, s));
    int64_t c = 0;
    TTG_RC(collect(mode, s, &c));
    *moved = 0;
    if (c == 0) return TTG_OK;
    limits_kernel<<<grid(k), 256, 0, stream>>>(k, mode, w.pw, b, w.room, w.want, w.spare, w.give);
    TTG_LAUNCH_CHECK();
    TTG_RC(admit(c, w.dest, w.room, w.want, w.ok_in, nullptr));
    TTG_RC(admit(c, part, w.spare, w.give, w.ok_out, nullptr));
    TTG_CUDA(cudaMemsetAsync(w.moved, 0, sizeof(unsigned long long), stream));
    apply_kernel<<<grid(c), 256, 0, stream>>>(c, w.order, w.ok_in, w.ok_out, w.dest, g.vw, part,
                                              (unsigned long long*)w.pw, w.moved);
    TTG_LAUNCH_CHECK();
    unsigned long long mv = 0;
    TTG_RC(read_back(&mv, w.moved, stream));
    *moved = (int64_t)mv;
    return TTG_OK;
  }

  int host_weights(std::vector<int64_t>& pw, bool* off) {
    pw.resize(k);
    TTG_CUDA(cudaMemcpyAsync(pw.data(), w.pw, sizeof(int64_t) * (size_t)k, cudaMemcpyDeviceToHost, stream));
    TTG_CUDA(cudaStreamSynchronize(stream));
    *off = false;
    for (int32_t p = 0; p < k; ++p) *off = *off || pw[p] > b.maxpw || pw[p] < b.minpw;
    return TTG_OK;
  }

  // exact fill: quotas on the host (what every part must give, what every part may take: deficits first, then
  // room), the leavers of every giving part by ascending internal connection, each sent to the part at its weight
  // offset in the concatenated quotas.  With unit vertex weights every part ends within its bounds.
  int fill(const std::vector<int64_t>& pw) {
    std::vector<int64_t> give(k, 0), tier(2 * (size_t)k, 0);
    int64_t out = 0, in = 0;
    for (int32_t p = 0; p < k; ++p) {
      give[p] = std::max<int64_t>(0, pw[p] - b.maxpw);
      tier[p] = std::max<int64_t>(0, b.minpw - pw[p]);
      out += give[p];
      in += tier[p];
    }
    for (int32_t p = 0; p < k && in > out; ++p) {   // more deficit than excess: parts above the lower bound donate
      if (pw[p] <= b.minpw) continue;
      const int64_t take = std::min(in - out, pw[p] - give[p] - b.minpw);
      if (take > 0) {
        give[p] += take;
        out += take;
      }
    }
    for (int32_t p = 0; p < k; ++p)
      tier[(size_t)k + p] = give[p] > 0 ? 0 : std::max<int64_t>(0, b.maxpw - pw[p] - tier[p]);
    for (size_t i = 1; i < tier.size(); ++i) tier[i] += tier[i - 1];
    TTG_CUDA(cudaMemcpyAsync(w.give, give.data(), sizeof(int64_t) * (size_t)k, cudaMemcpyHostToDevice, stream));
    TTG_CUDA(cudaMemcpyAsync(w.cum, tier.data(), sizeof(int64_t) * tier.size(), cudaMemcpyHostToDevice, stream));
    limits_kernel<<<grid(k), 256, 0, stream>>>(k, M_FILL, w.pw, b, w.room, w.want, w.spare, w.give);
    TTG_LAUNCH_CHECK();
    fill_cand_kernel<<<grid(g.n * 32), 256, 0, stream>>>(g.n, g.xadj, g.adj, g.adjw, part, w.give, w.internal,
                                                          w.cand);
    TTG_LAUNCH_CHECK();
    const uint64_t s = salt();
    int64_t c = 0;
    TTG_RC(collect(M_FILL, s, &c));   // blocks until the quotas above are on the device
    if (c == 0) return TTG_OK;
    int32_t* grouped = nullptr;
    TTG_RC(admit(c, part, w.spare, w.give, w.ok_out, &grouped));
    return fill_apply(c, grouped);
  }

  int fill_apply(int64_t c, const int32_t* grouped);
};

// ok_out is indexed by vertex; the leavers keep the grouped order
__global__ void __launch_bounds__(256)
gather_flags_kernel(int64_t c, const int32_t* __restrict__ grouped, const uint8_t* __restrict__ ok_v,
                    uint8_t* __restrict__ ok_i) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < c) ok_i[i] = ok_v[grouped[i]];
}

int Refine::fill_apply(int64_t c, const int32_t* grouped) {
  // flags by position (ok_in is free here), then the order-preserving selection of the leavers
  gather_flags_kernel<<<grid(c), 256, 0, stream>>>(c, grouped, w.ok_out, w.ok_in);
  TTG_LAUNCH_CHECK();
  size_t bytes = w.cub_bytes;
  TTG_CUDA(cub::DeviceSelect::Flagged(w.cub_tmp, bytes, grouped, w.ok_in, w.list, w.counts, c, stream));
  count_launch();
  int32_t leavers = 0;
  TTG_RC(read_back(&leavers, w.counts, stream));
  if (leavers == 0) return TTG_OK;
  weights_kernel<<<grid(leavers), 256, 0, stream>>>(leavers, w.list, g.vw, w.excl);
  TTG_LAUNCH_CHECK();
  bytes = w.cub_bytes;
  TTG_CUDA(cub::DeviceScan::ExclusiveSum(w.cub_tmp, bytes, w.excl, w.excl, (int64_t)leavers, stream));
  count_launch();
  fill_dest_kernel<<<grid(leavers), 256, 0, stream>>>(leavers, k, w.list, w.excl, w.cum, w.dest, w.ok_in);
  TTG_LAUNCH_CHECK();
  TTG_CUDA(cudaMemsetAsync(w.moved, 0, sizeof(unsigned long long), stream));
  apply_kernel<<<grid(leavers), 256, 0, stream>>>(leavers, w.list, w.ok_in, w.ok_in, w.dest, g.vw, part,
                                                  (unsigned long long*)w.pw, w.moved);
  TTG_LAUNCH_CHECK();
  return TTG_OK;
}

}  // namespace
}  // namespace ttg

using namespace ttg;

extern "C" size_t ttg_kway_symmetrise_workspace_bytes(int64_t num_nodes, int64_t num_edges) {
  if (!nodes_in_range(num_nodes) || !edges_in_range(num_edges)) return 0;
  return carve_sym(nullptr, num_nodes, num_edges).total;
}

extern "C" int ttg_kway_symmetrise(int64_t num_nodes, int64_t num_edges, const int64_t* indptr, const int32_t* indices,
                                   int64_t* xadj, int32_t* adj, int32_t* adjw, int32_t* vw, int64_t* sym_edges_out,
                                   void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  TTG_CHECK_ARG(nodes_in_range(num_nodes), "kway_symmetrise: num_nodes=%lld out of range", (long long)num_nodes);
  TTG_CHECK_ARG(edges_in_range(num_edges), "kway_symmetrise: num_edges=%lld out of range", (long long)num_edges);
  TTG_CHECK_ARG(indptr && (indices || num_edges == 0) && xadj && adj && adjw && vw && sym_edges_out,
                "kway_symmetrise: null pointer");
  SymWs w = carve_sym(workspace, num_nodes, num_edges);
  if (!workspace || workspace_bytes < w.total) {
    set_error("kway_symmetrise: workspace %zu bytes, need %zu for %lld nodes / %lld edges", workspace_bytes, w.total,
              (long long)num_nodes, (long long)num_edges);
    return TTG_ENOMEM;
  }
  const int64_t n = num_nodes, items = 2 * num_edges;
  const int colbits = std::max(1, bits_for((uint64_t)(n - 1)));
  const uint64_t drop = 1ull << (2 * colbits);
  TTG_CUDA(cudaMemsetAsync(w.flags, 0, sizeof(int32_t), stream));
  fill_i32_kernel<<<grid(n), 256, 0, stream>>>(n, 1, vw);
  TTG_LAUNCH_CHECK();
  if (num_edges == 0) {
    TTG_CUDA(cudaMemsetAsync(xadj, 0, sizeof(int64_t) * (size_t)(n + 1), stream));
    *sym_edges_out = 0;
    return TTG_OK;
  }
  const int64_t counts0[2] = {n, 0};
  TTG_CUDA(cudaMemcpyAsync(w.counts, counts0, sizeof(counts0), cudaMemcpyHostToDevice, stream));
  sym_emit_kernel<<<grid(n * 32), 256, 0, stream>>>(n, num_edges, colbits, drop, indptr, indices, w.keys_a, w.flags);
  TTG_LAUNCH_CHECK();
  cub::DoubleBuffer<uint64_t> dk(w.keys_a, w.keys_b);
  size_t bytes = w.cub_bytes;
  TTG_CUDA(cub::DeviceRadixSort::SortKeys(w.cub_tmp, bytes, dk, items, 0, 2 * colbits + 1, stream));
  count_launch();
  int32_t bad = 0;
  TTG_RC(read_back(&bad, w.flags, stream));
  if (bad) {
    set_error("kway_symmetrise: an in-neighbour id lies outside [0, %lld) or indptr is not a CSR of %lld edges",
              (long long)n, (long long)num_edges);
    return TTG_EINVAL;
  }
  TTG_RC(keys_to_csr(items, colbits, drop, dk, nullptr, n, w.pos, w.counts, w.cub_tmp, w.cub_bytes, xadj, adj, adjw,
                     stream));
  return read_back(sym_edges_out, w.counts + 1, stream);
}

extern "C" size_t ttg_kway_coarsen_workspace_bytes(int64_t num_nodes, int64_t num_edges) {
  if (!nodes_in_range(num_nodes) || !edges_in_range(num_edges)) return 0;
  return carve_coarsen(nullptr, num_nodes, num_edges).total;
}

extern "C" int ttg_kway_coarsen(int64_t num_nodes, int64_t num_edges, const int64_t* xadj, const int32_t* adj,
                                const int32_t* adjw, const int32_t* vw, int32_t maxvw, uint64_t seed, int32_t level,
                                int32_t* cmap, int64_t* cxadj, int32_t* cadj, int32_t* cadjw, int32_t* cvw,
                                int64_t* counts_out, void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  TTG_CHECK_ARG(nodes_in_range(num_nodes), "kway_coarsen: num_nodes=%lld out of range", (long long)num_nodes);
  TTG_CHECK_ARG(edges_in_range(num_edges), "kway_coarsen: num_edges=%lld out of range", (long long)num_edges);
  TTG_CHECK_ARG(maxvw >= 1, "kway_coarsen: maxvw=%d below 1", maxvw);
  TTG_CHECK_ARG(xadj && (num_edges == 0 || (adj && adjw)) && vw && cmap && cxadj && (num_edges == 0 || (cadj && cadjw)) &&
                    cvw && counts_out,
                "kway_coarsen: null pointer");
  CoarsenWs w = carve_coarsen(workspace, num_nodes, num_edges);
  if (!workspace || workspace_bytes < w.total) {
    set_error("kway_coarsen: workspace %zu bytes, need %zu for %lld nodes / %lld edges", workspace_bytes, w.total,
              (long long)num_nodes, (long long)num_edges);
    return TTG_ENOMEM;
  }
  const int64_t n = num_nodes, m = num_edges;
  const uint64_t lseed = mix64(seed ^ mix64(0x636f6172ull + (uint64_t)level));
  // handshake matching
  fill_i32_kernel<<<grid(n), 256, 0, stream>>>(n, -1, w.match);
  TTG_LAUNCH_CHECK();
  for (int r = 0; r < kMatchRounds && m > 0; ++r) {
    match_propose_kernel<<<grid(n * 32), 256, 0, stream>>>(n, xadj, adj, adjw, vw, maxvw, w.match, w.prop,
                                                           mix64(lseed + (uint64_t)r));
    TTG_LAUNCH_CHECK();
    match_accept_kernel<<<grid(n), 256, 0, stream>>>(n, w.prop, w.match);
    TTG_LAUNCH_CHECK();
  }
  // two-hop pass and isolated vertices
  twohop_key_kernel<<<grid(n), 256, 0, stream>>>(n, xadj, adj, adjw, w.match, w.hkeys_a);
  TTG_LAUNCH_CHECK();
  cub::DoubleBuffer<uint64_t> hk(w.hkeys_a, w.hkeys_b);
  size_t bytes = w.cub_bytes;
  TTG_CUDA(cub::DeviceRadixSort::SortKeys(w.cub_tmp, bytes, hk, n, 0, 64, stream));
  count_launch();
  twohop_start_kernel<<<grid(n), 256, 0, stream>>>(n, hk.Current(), w.start);
  TTG_LAUNCH_CHECK();
  bytes = w.cub_bytes;
  TTG_CUDA(cub::DeviceScan::InclusiveScan(w.cub_tmp, bytes, w.start, w.start, cub::Max(), n, stream));
  count_launch();
  twohop_pair_kernel<<<grid(n), 256, 0, stream>>>(n, hk.Current(), w.start, vw, maxvw, w.match);
  TTG_LAUNCH_CHECK();
  // coarse ids
  leader_kernel<<<grid(n), 256, 0, stream>>>(n, w.match, w.lead);
  TTG_LAUNCH_CHECK();
  bytes = w.cub_bytes;
  TTG_CUDA(cub::DeviceScan::ExclusiveSum(w.cub_tmp, bytes, w.lead, w.id, n, stream));
  count_launch();
  cmap_kernel<<<grid(n), 256, 0, stream>>>(n, w.match, w.lead, w.id, vw, cmap, cvw, w.counts);
  TTG_LAUNCH_CHECK();
  // contraction
  const int colbits = std::max(1, bits_for((uint64_t)(n - 1)));
  const uint64_t drop = 1ull << (2 * colbits);
  if (m > 0) {
    contract_emit_kernel<<<grid(n * 32), 256, 0, stream>>>(n, colbits, drop, xadj, adj, adjw, cmap, w.keys_a, w.w_a);
    TTG_LAUNCH_CHECK();
    cub::DoubleBuffer<uint64_t> dk(w.keys_a, w.keys_b);
    cub::DoubleBuffer<int32_t> dv(w.w_a, w.w_b);
    bytes = w.cub_bytes;
    TTG_CUDA(cub::DeviceRadixSort::SortPairs(w.cub_tmp, bytes, dk, dv, m, 0, 2 * colbits + 1, stream));
    count_launch();
    TTG_RC(keys_to_csr(m, colbits, drop, dk, dv.Current(), n, w.pos, w.counts, w.cub_tmp, w.cub_bytes, cxadj, cadj,
                       cadjw, stream));
  } else {
    TTG_CUDA(cudaMemsetAsync(w.counts + 1, 0, sizeof(int64_t), stream));
    TTG_CUDA(cudaMemsetAsync(cxadj, 0, sizeof(int64_t) * (size_t)(n + 1), stream));
  }
  TTG_CUDA(cudaMemcpyAsync(counts_out, w.counts, 2 * sizeof(int64_t), cudaMemcpyDeviceToHost, stream));
  TTG_CUDA(cudaStreamSynchronize(stream));
  return TTG_OK;
}

extern "C" size_t ttg_kway_refine_workspace_bytes(int64_t num_nodes, int32_t k) {
  if (!nodes_in_range(num_nodes) || k < 1 || k > num_nodes) return 0;
  return carve_refine(nullptr, num_nodes, k).total;
}

extern "C" int ttg_kway_refine(int64_t num_nodes, const int64_t* xadj, const int32_t* adj, const int32_t* adjw,
                               const int32_t* vw, int64_t total_nodes, int32_t k, float ubfactor, int32_t finest,
                               uint64_t seed, int32_t level, int32_t refine_passes, const int32_t* cmap,
                               const int32_t* coarse_part, int32_t* part, int64_t* stats_out, void* workspace,
                               size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  TTG_CHECK_ARG(nodes_in_range(num_nodes) && num_nodes <= total_nodes && total_nodes < (int64_t)INT32_MAX,
                "kway_refine: %lld of %lld nodes out of range", (long long)num_nodes, (long long)total_nodes);
  TTG_CHECK_ARG(k >= 1 && k <= num_nodes, "kway_refine: k=%d for %lld nodes", k, (long long)num_nodes);
  TTG_CHECK_ARG(ubfactor >= 1.0f, "kway_refine: ubfactor %g below 1", (double)ubfactor);
  TTG_CHECK_ARG(xadj && vw && part && (cmap == nullptr) == (coarse_part == nullptr), "kway_refine: null pointer");
  RefineWs ws = carve_refine(workspace, num_nodes, k);
  if (!workspace || workspace_bytes < ws.total) {
    set_error("kway_refine: workspace %zu bytes, need %zu for %lld nodes / k = %d", workspace_bytes, ws.total,
              (long long)num_nodes, (long long)k);
    return TTG_ENOMEM;
  }
  if (refine_passes <= 0) refine_passes = 10;
  KwayBounds kb;
  kway_bounds(total_nodes, k, ubfactor, &kb);
  Refine r;
  r.g = Level{num_nodes, xadj, adj, adjw, vw};
  r.k = k;
  r.b = finest ? Bounds{kb.maxpw, kb.minpw} : Bounds{kb.maxpw_coarse, kb.minpw_coarse};
  r.seed = mix64(seed ^ mix64(0x726566ull + (uint64_t)level));
  r.part = part;
  r.w = ws;
  r.stream = stream;
  const int64_t n = num_nodes;
  if (cmap) {
    project_kernel<<<grid(n), 256, 0, stream>>>(n, cmap, coarse_part, part);
    TTG_LAUNCH_CHECK();
  }
  TTG_CUDA(cudaMemsetAsync(ws.counts, 0, 4 * sizeof(int32_t), stream));
  heavy_list_kernel<<<grid(n), 256, 0, stream>>>(n, xadj, ws.heavy, ws.counts + 1);
  TTG_LAUNCH_CHECK();
  TTG_RC(r.part_weights());
  int32_t c4[4];
  TTG_CUDA(cudaMemcpyAsync(c4, ws.counts, sizeof(c4), cudaMemcpyDeviceToHost, stream));
  TTG_CUDA(cudaStreamSynchronize(stream));
  if (c4[2]) {
    set_error("kway_refine: a part id lies outside [0, %d)", k);
    return TTG_EINVAL;
  }
  r.heavy = c4[1];
  std::vector<int64_t> pw;
  int64_t rebalance_rounds = 0, iterations = 0, fills = 0;
  // rebalance: moves to adjacent parts first; what they leave goes through the exact fill
  auto rebalance = [&]() -> int {
    bool off = false;
    for (int round = 0; round < kLocalRebalanceRounds; ++round) {
      TTG_RC(r.host_weights(pw, &off));
      if (!off) return TTG_OK;
      int64_t moved = 0;
      TTG_RC(r.round(M_REBALANCE, &moved));
      ++rebalance_rounds;
      if (moved == 0) break;
    }
    for (int f = 0; f < 3; ++f) {
      TTG_RC(r.host_weights(pw, &off));
      if (!off) return TTG_OK;
      TTG_RC(r.fill(pw));
      ++fills;
    }
    TTG_RC(r.host_weights(pw, &off));
    if (off && finest) {
      set_error("kway_refine: the balance bound [%lld, %lld] was not met", (long long)r.b.minpw,
                (long long)r.b.maxpw);
      return TTG_EINVAL;
    }
    return TTG_OK;
  };
  TTG_RC(rebalance());
  for (int it = 0; it < kItersPerPass * refine_passes; ++it) {
    int64_t moved = 0;
    TTG_RC(r.round(M_REFINE, &moved));
    ++iterations;
    if (moved == 0) break;
  }
  TTG_RC(rebalance());
  if (stats_out) {
    stats_out[0] = iterations;
    stats_out[1] = rebalance_rounds;
    stats_out[2] = fills;
  }
  return TTG_OK;
}

extern "C" size_t ttg_kway_edge_cut_workspace_bytes(void) { return 256; }

extern "C" int ttg_kway_edge_cut(int64_t num_nodes, const int64_t* indptr, const int32_t* indices, const int32_t* part,
                                 int64_t* cut_out, void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  TTG_CHECK_ARG(nodes_in_range(num_nodes), "kway_edge_cut: num_nodes=%lld out of range", (long long)num_nodes);
  TTG_CHECK_ARG(indptr && indices && part && cut_out, "kway_edge_cut: null pointer");
  if (!workspace || workspace_bytes < 256) {
    set_error("kway_edge_cut: workspace %zu bytes, need 256", workspace_bytes);
    return TTG_ENOMEM;
  }
  unsigned long long* cut = (unsigned long long*)workspace;
  TTG_CUDA(cudaMemsetAsync(cut, 0, sizeof(*cut), stream));
  cut_kernel<<<grid(num_nodes * 32), 256, 0, stream>>>(num_nodes, indptr, indices, part, cut);
  TTG_LAUNCH_CHECK();
  return read_back(cut_out, (const int64_t*)cut, stream);
}
