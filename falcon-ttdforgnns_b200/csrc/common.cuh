// common.cuh -- shared helpers for the ttg_b200 kernels (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/ttg_b200.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "ttg_b200 is written for sm_100a (B200) only"
#endif

namespace ttg {

constexpr int kWarp = 32;
constexpr int kNumSMs = 148;  // B200: 2 dies x 74 SMs

// ---- error plumbing (host) ---------------------------------------------------------
void set_error(const char* fmt, ...);
void count_launch(int n = 1);

#define TTG_CHECK_ARG(cond, ...)  \
  do {                            \
    if (!(cond)) {                \
      ttg::set_error(__VA_ARGS__); \
      return TTG_EINVAL;          \
    }                             \
  } while (0)

#define TTG_CUDA(expr)                                                              \
  do {                                                                              \
    cudaError_t _e = (expr);                                                        \
    if (_e != cudaSuccess) {                                                        \
      ttg::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr,                  \
                     cudaGetErrorString(_e));                                       \
      return TTG_ECUDA;                                                             \
    }                                                                               \
  } while (0)

#define TTG_LAUNCH_CHECK()                                                          \
  do {                                                                              \
    ttg::count_launch();                                                            \
    cudaError_t _e = cudaGetLastError();                                            \
    if (_e != cudaSuccess) {                                                        \
      ttg::set_error("%s:%d: kernel launch -> %s", __FILE__, __LINE__,              \
                     cudaGetErrorString(_e));                                       \
      return TTG_ECUDA;                                                             \
    }                                                                               \
  } while (0)

// opt-in to more than 48 KB of dynamic shared memory, once per kernel AND device (the attribute
// belongs to the device's context; a process may drive several GPUs)
#define TTG_ENSURE_SMEM(kern, bytes)                                                          \
  do {                                                                                        \
    static size_t _ttg_set[32] = {};                                                          \
    int _ttg_dev = 0;                                                                         \
    TTG_CUDA(cudaGetDevice(&_ttg_dev));                                                       \
    const bool _ttg_in = _ttg_dev >= 0 && _ttg_dev < 32;                                      \
    if (!_ttg_in || _ttg_set[_ttg_dev] < (size_t)(bytes)) {                                   \
      TTG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,        \
                                    (int)(bytes)));                                           \
      if (_ttg_in) _ttg_set[_ttg_dev] = (size_t)(bytes);                                      \
    }                                                                                         \
  } while (0)

// ---- optional per-kernel timing (CUDA events on the launching stream), api.cu ------------
enum KernelId {
  K_PLAN = 0, K_SORT, K_ZERO_ROWS, K_FWD, K_BWD_ROWS, K_BWD_CORES, K_REDUCE, K_OPTIM,
  K_GENERIC_FWD, K_GENERIC_BWD, K_TABLE, K_COUNT
};
void prof_begin(int id, cudaStream_t s);
void prof_end(int id, cudaStream_t s);

// ---- device-side view of a TT table (passed by value as a kernel parameter) ---------
struct TTDev {
  int32_t T;
  int32_t num_tables;
  int32_t D;                         // prod(q)
  int32_t p[TTG_MAX_CORES];
  int32_t q[TTG_MAX_CORES];
  int32_t r[TTG_MAX_CORES + 1];
  int32_t cols[TTG_MAX_CORES];       // r[t]*q[t]*r[t+1]
  int64_t L[TTG_MAX_CORES];          // prod(p[t+1:])
  int64_t num_rows;                  // prod(p)
  float* core[TTG_MAX_CORES];        // device pointers [num_tables][p[t]][cols[t]]
};

// Validates `shape` and fills `dev` (host). Returns TTG_OK / TTG_EINVAL.
int make_ttdev(const ttg_shape* shape, const float* const* host_core_ptrs, TTDev* dev);

static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }
static inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

// number of bits that hold every value in [0, x] (radix-sort key widths)
static inline int bits_for(uint64_t x) {
  int b = 0;
  while (b < 64 && (x >> b) != 0) ++b;
  return b;
}

// lays a caller's workspace out in 256-byte aligned pieces; with base == nullptr it only sums the sizes
struct Carver {
  void* base;
  size_t off = 0;
  void* take(size_t bytes) {
    char* p = base ? (char*)base + off : nullptr;
    off += align_up(bytes, 256);
    return (void*)p;
  }
};

// one value from the device, waited for
template <typename T>
int read_back(T* host, const T* dev, cudaStream_t stream) {
  TTG_CUDA(cudaMemcpyAsync(host, dev, sizeof(T), cudaMemcpyDeviceToHost, stream));
  TTG_CUDA(cudaStreamSynchronize(stream));
  return TTG_OK;
}

#define TTG_RC(expr)               \
  do {                             \
    const int _rc = (expr);        \
    if (_rc != TTG_OK) return _rc; \
  } while (0)

// ---- device helpers ------------------------------------------------------------------
__device__ __forceinline__ float4 ldg4(const float* p) {
  return __ldg(reinterpret_cast<const float4*>(p));
}
__device__ __forceinline__ void red_add_v4(float* p, float4 v) {
  // REDG.E.ADD.F32x4 : one 16-byte reduction instead of four scalar atomics
  asm volatile("red.global.add.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y),
               "f"(v.z), "f"(v.w)
               : "memory");
}
__device__ __forceinline__ void st_cs_v4(float* p, float4 v) {
  // streaming store: written once, not re-read by this kernel
  asm volatile("st.global.cs.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y),
               "f"(v.z), "f"(v.w)
               : "memory");
}

// ---- programmatic dependent launch ----------------------------------------------------------
// A kernel launched with launch_pdl may start while the kernel before it on the stream is still
// running (as soon as all its CTAs have executed pdl_trigger or exited); everything it does before
// pdl_wait() must be independent of that kernel (shared-memory staging of operands nobody is
// writing).  pdl_wait() returns once the preceding kernel has completed and its writes are
// visible.  Both instructions are no-ops in a launch without the attribute.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
// After pdl_wait(), data that a preceding kernel of the chain produced must NOT be read with
// __ldg / through const __restrict__ pointers: those become ld.global.nc, which both the compiler
// and ptxas treat as invariant and hoist above griddepcontrol.wait when the address is known early
// (ptxas did: the backward row kernel read the plan's row count before the scan kernel of the same
// call had written it -- wrong gradients whenever the previous call had a different count).  The
// ld_dep_* loads below are ordinary ld.global in volatile asm: ordered after the wait, and every
// load whose address depends on their result is ordered behind them by that dependence.
__device__ __forceinline__ uint32_t ld_dep_u32(const void* p) {
  uint32_t v;
  asm volatile("ld.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ int32_t ld_dep_s32(const void* p) { return (int32_t)ld_dep_u32(p); }
__device__ __forceinline__ float ld_dep_f32(const void* p) {
  float v;
  asm volatile("ld.global.f32 %0, [%1];" : "=f"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ int4 ld_dep_int4(const void* p) {
  int4 v;
  asm volatile("ld.global.v4.s32 {%0,%1,%2,%3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
               : "l"(p)
               : "memory");
  return v;
}
__device__ __forceinline__ float4 ld_dep_float4(const void* p) {
  float4 v;
  asm volatile("ld.global.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "l"(p)
               : "memory");
  return v;
}

int pdl_level();   // api.cu: environment TTG_PDL_LEVEL, default 1
                   // 0: ordinary launches; 1: row / cores / finalize kernels; 2: also the plan chain
                   // (scan, scatter, table).  Level 2 is correct (full suite) but gains nothing
                   // measurable over level 1, so it stays opt-in.

template <int LEVEL = 1, typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem,
                              cudaStream_t stream, Args... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = (pdl_level() >= LEVEL) ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}

// ---- internal entry points shared between translation units --------------------------
// generic (any T) kernels, tt_generic.cu
int generic_forward(const TTDev& tt, int64_t B, int64_t nnz, const int64_t* indices,
                    const int64_t* rowidx, const int64_t* tableidx, float* output,
                    cudaStream_t stream);
int generic_backward(const TTDev& tt, int64_t B, int64_t nnz, const int64_t* indices,
                     const int64_t* rowidx, const int64_t* tableidx, const float* d_output,
                     float* const* dcore, cudaStream_t stream);
// optimizer over whole cores, tt_generic.cu
int apply_optimizer(const TTDev& tt, int32_t optim, float lr, float eps, float* const* dcore,
                    float* const* state, cudaStream_t stream);

// sorted prefix-reuse kernels for T == 3, tt_sorted.cu
bool sorted_supported(const TTDev& tt);
size_t sorted_workspace_bytes(const TTDev& tt, int64_t B, int64_t nnz);
int sorted_forward(const TTDev& tt, int64_t B, int64_t nnz, const int64_t* indices,
                   const int64_t* rowidx, const int64_t* tableidx, float* output, void* ws,
                   size_t ws_bytes, int32_t flags, cudaStream_t stream);
// dense gradients into dcore AND the optimizer step (optim/lr/eps/state), fused in the last kernel
int sorted_backward(const TTDev& tt, int64_t B, int64_t nnz, const int64_t* indices,
                    const int64_t* rowidx, const int64_t* tableidx, const float* d_output,
                    float* const* dcore, int32_t optim, float lr, float eps, float* const* state,
                    void* ws, size_t ws_bytes, int32_t flags, cudaStream_t stream);

int sorted_plan(const TTDev& tt, int64_t B, int64_t nnz, const int64_t* indices, const int64_t* rowidx,
                const int64_t* tableidx, void* ws, size_t ws_bytes, int32_t flags, cudaStream_t stream);

int sorted_rows_range(const TTDev& tt, int64_t first_row, int64_t num, float* output, void* ws,
                      size_t ws_bytes, int32_t flags, cudaStream_t stream);

// tensor-core kernels for the group-table strategy, tt_mma.cu (plan built by tt_sorted.cu)
struct MmaPlan {
  const uint32_t* skeys;   // keys grouped by (i0, i1), invalid keys last
  const int32_t* srow;     // output row of each sorted key, bit 31 = bag has several indices
  const int32_t* cnt;      // [groups + 1] rows per group (last: invalid keys)
  const int32_t* base;     // [groups + 1] exclusive scan of cnt
  float* Ttab;             // [groups][q0 q1][r2]
  float* S;                // [groups][q0 q1][r2]
  float* d0parts;          // [p1][core0 elements]: per-i1 partial products of d_core0
  uint32_t first_key;      // skeys == nullptr: the keys are first_key, first_key + 1, ...
  int32_t spare_sms;       // SMs the persistent row kernels leave to other streams (TTG_FLAG_SHARE_SMS)
};
bool mma_supported(const TTDev& tt);       // table, forward and backward
bool mma_fwd_supported(const TTDev& tt);   // table and forward (ranks 32: the backward stays FFMA)
int mma_table(const TTDev& tt, const MmaPlan& pl, bool tf32, bool chained, cudaStream_t stream);
int mma_forward(const TTDev& tt, int64_t nnz, uint32_t total_rows, const MmaPlan& pl, float* output,
                bool tf32, cudaStream_t stream);
int mma_backward(const TTDev& tt, int64_t nnz, uint32_t total_rows, const MmaPlan& pl,
                 const float* d_output, float* const* dcore, int32_t optim, float lr, float eps,
                 float* const* state, bool tf32, cudaStream_t stream);

// the two dense reductions over S (d_core1, d_core0) + optimizer, for an S any row kernel wrote
// (d_core2 must be complete): ranks 32 pair the FFMA row kernel with these
int mma_cores_finalize(const TTDev& tt, const MmaPlan& pl, float* const* dcore, int32_t optim, float lr,
                       float eps, float* const* state, bool tf32, cudaStream_t stream);

// right-grouped kernels on the sm_100a tensor path (tcgen05 + TMEM), tt_tc5.cu.  The plan is the one of
// tt_sorted.cu built on TRANSPOSED keys  table * prod(p) + (idx % (p1 p2)) * p0 + idx / (p1 p2):
// group = key / p0 = (table, i1, i2), i0 = key % p0.
struct RPlan {
  const uint32_t* skeys;
  const int32_t* srow;
  const int32_t* cnt;      // [groups + 1] rows per group
  const int32_t* base;     // [groups + 1] exclusive scan
  float* tab;              // [groups][2][r1 * q1 q2]  tr1 operand images, hi plane then lo plane
  float* S1;               // [groups][r1][q1 q2]      d(tr1), written by the backward row kernel
  float* d0parts;          // [kNumSMs][core0 elements] per-CTA copies of d_core0
  float* d2parts;          // [tables][p1][p2][r2 q2]  d_core2 per i1 (right-grouped mma.sync cores kernel)
};
bool r_supported(const TTDev& tt);
size_t r_table_floats(const TTDev& tt);
// planes: 2 = operand image and its TF32 remainder (tcgen05 kernels), 1 = the image only (mma.sync kernels)
int r_table(const TTDev& tt, const RPlan& pl, int planes, cudaStream_t stream);
int r_forward(const TTDev& tt, int64_t nnz, const RPlan& pl, float* output, bool tf32, cudaStream_t stream);
int r_backward(const TTDev& tt, int64_t nnz, const RPlan& pl, const float* d_output, float* const* dcore,
               int32_t optim, float lr, float eps, float* const* state, bool tf32, cudaStream_t stream);
// the same path on mma.sync (warp-level tensor cores), tt_rmma.cu
int rm_forward(const TTDev& tt, int64_t nnz, const RPlan& pl, float* output, bool tf32, cudaStream_t stream);
int rm_backward(const TTDev& tt, int64_t nnz, const RPlan& pl, const float* d_output, float* const* dcore,
                int32_t optim, float lr, float eps, float* const* state, bool tf32, cudaStream_t stream);
bool rm_supported(const TTDev& tt);
// d_core1 / d_core2 from S1 (tt_tc5.cu)
int r_cores(const TTDev& tt, const RPlan& pl, float* const* dcore, cudaStream_t stream);
// d_core0 = sum of `nparts` partial copies (fixed order) + optimizer step on all three cores, tt_mma.cu
// (+ d_core2 = sum over its n2parts copies per table when d2parts is given)
int mma_finalize_parts(const TTDev& tt, const float* d0parts, int nparts, const float* d2parts, int n2parts,
                       float* const* dcore, int32_t optim, float lr, float eps, float* const* state,
                       cudaStream_t stream);

// balance bounds of the k-way partitioners (kway_host.cu): every part at most maxpw and at least minpw vertices
// on the finest level, maxpw_coarse / minpw_coarse (1.3 x slack) on the coarser ones
struct KwayBounds {
  int64_t maxpw, minpw, maxpw_coarse, minpw_coarse;
};
void kway_bounds(int64_t num_nodes, int32_t k, float ubfactor, KwayBounds* b);

}  // namespace ttg
