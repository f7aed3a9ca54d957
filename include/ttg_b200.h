/*
 * ttg_b200.h -- C ABI of the B200-native TT-embedding hot path.
 *
 * This is the drop-in boundary: every entry point below replaces one function of the
 * reference's pybind modules (the citation after "replaces:" is path:line relative to the
 * reference tree).  Plain pointers and sizes only: no ATen/torch types, no allocation, no
 * hidden state.  All pointers are DEVICE pointers unless a parameter is named host_*.
 * Every call enqueues work on `stream` (a cudaStream_t passed as void*) and returns
 * without synchronising, except ttg_preprocess_indices whose contract is to return the
 * host integer nnz_tt (the reference synchronises there too,
 * FBTT/tt_embeddings_cuda.cu:1492-1499).
 *
 * Return value: 0 on success, a negative TTG_E* code otherwise; ttg_last_error() gives the
 * message of the last failure on the calling thread.  The Python shim turns a non-zero
 * return into RuntimeError, which is what TORCH_CHECK does in the reference
 * (FBTT/tt_embeddings_cuda.cu:991-994).
 *
 * Layout conventions (identical to the reference, FBTT/tt_embeddings_ops.py:519-545):
 *   core t   : fp32 [num_tables][p[t]][r[t]*q[t]*r[t+1]], row i_t is the row-major matrix
 *              [r[t]][q[t]][r[t+1]]
 *   L        : int64 [T], L[t] = prod(p[t+1:])     index split i_t = (idx % L[t-1]) / L[t]
 *   output   : fp32 [num_tables][B][D], D = prod(q)
 *   indices, rowidx, tableidx : int64 [nnz]
 */
#ifndef TTG_B200_H_
#define TTG_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TTG_MAX_CORES 4
#define TTG_MAX_PEERS 8           /* GPUs of one NVSwitch node                  */
#define TTG_PEER_HANDLE_BYTES 64   /* sizeof(cudaIpcMemHandle_t)                 */

enum {
  TTG_OK = 0,
  TTG_EINVAL = -1,   /* bad argument (shape, null pointer, D % 4 != 0 ...) */
  TTG_ECUDA = -2,    /* a CUDA runtime call or kernel launch failed          */
  TTG_ENOMEM = -3,   /* workspace too small                                  */
  TTG_ENOTSUP = -4   /* shape outside what the kernels support               */
};

enum { TTG_OPTIM_SGD = 0, TTG_OPTIM_ADAGRAD = 1, TTG_OPTIM_DENSE = 2 };

/* flags for ttg_tt_forward / ttg_tt_backward */
enum {
  TTG_FLAG_FORCE_GENERIC = 1, /* use the shape-generic kernels (any T in 2..4)      */
  TTG_FLAG_PLAN_VALID = 2,    /* workspace already holds the index plan (and group table) of
                                 the SAME (indices, rowidx, nnz, B) and the cores have not
                                 changed since -- skip both (forward -> backward reuse)   */
  TTG_FLAG_DETERMINISTIC = 4, /* full radix sort instead of the bucket plan: fixed summation
                                 order for d_core0 / d_core1 run to run                */
  TTG_FLAG_TF32 = 8,          /* tensor-core kernels use plain TF32 operands (about 1e-3
                                 relative) instead of the default 3xTF32 split, which keeps
                                 fp32 accuracy (about 3e-7 relative)                    */
  TTG_FLAG_FFMA = 16,         /* fp32 FFMA kernels instead of the tensor-core kernels     */
  TTG_FLAG_MMA_SYNC = 32,     /* force the mma.sync (warp-level) tensor-core kernels: the default,
                                 the flag exists so that a caller can name it           */
  TTG_FLAG_PLAN_READY = 128,  /* forward: the workspace slot holds the index plan ttg_tt_plan built for
                                 the SAME (indices, rowidx, tableidx, nnz, B); only the group table is
                                 still computed (it depends on the cores)              */
  TTG_FLAG_PLAN_SLOT1 = 256,  /* use the second of the two plan slots of the workspace (ttg_tt_plan,
                                 forward and backward of one batch must name the same slot) */
  TTG_FLAG_SHARE_SMS = 512,   /* the persistent row kernels leave 8 of the 148 SMs to other streams (a CTA
                                 of theirs takes a whole register file, so nothing co-resides with them):
                                 for callers that run ttg_tt_plan, a sampler or copies beside a step */
  TTG_FLAG_RIGHT = 1024,      /* the right-grouped mma.sync kernels (csrc/tt_rmma.cu; q0 = 4, ranks 16,16, batch
                                 dense in (i1, i2) groups): groups (i1, i2), tr1 = core1 core2 from a table.
                                 Without this flag they are used from 14 rows per (i1, i2) group and call on
                                 (274,400 rows at products shape: cheaper per row, dearer per group;
                                 DESIGN.md section 4c); TTG_FLAG_MMA_SYNC keeps the
                                 left-grouped kernels at any size */
  TTG_FLAG_TCGEN05 = 64       /* the tcgen05 / tensor-memory kernels (csrc/tt_tc5.cu; q0 = 4, ranks
                                 16,16, batch dense in (i1, i2) groups): same results, measured
                                 slower than the mma.sync kernels on B200 at the BASELINE batch
                                 (DESIGN.md section 4b), hence opt-in                    */
};

/* TT table description: tt_p_shapes / tt_q_shapes / tt_ranks of the reference. */
typedef struct ttg_shape {
  int32_t T;                      /* number of cores, 2..4                      */
  int32_t num_tables;             /* tt_cores[t].size(0)                        */
  int32_t p[TTG_MAX_CORES];       /* tt_p_shapes                                */
  int32_t q[TTG_MAX_CORES];       /* tt_q_shapes                                */
  int32_t r[TTG_MAX_CORES + 1];   /* tt_ranks incl. the leading/trailing 1      */
} ttg_shape;

const char* ttg_last_error(void);
int ttg_version(void);
/* number of kernel launches issued by this library on the calling process so far */
int64_t ttg_launch_count(void);

/* Per-kernel timing for bench.py's roofline line: when enabled, the library brackets each of
 * its main kernels with CUDA events on the launching stream (do not enable while capturing a
 * CUDA graph).  ttg_profile_read synchronises on the recorded events and returns the total
 * device time and launch count of kernel class `id` since the last enable; ttg_profile_name
 * returns its name or NULL when id is out of range. */
int ttg_profile_enable(int32_t on);
int ttg_profile_read(int32_t id, double* total_ms, int64_t* count);
const char* ttg_profile_name(int32_t id);

/* ------------------------------------------------------------------------------------
 * (a) TT chain contraction: forward.
 * replaces: tt_embeddings_forward_cuda  FBTT/tt_embeddings_cuda.cu:967-1081 (op tt_forward,
 *           FBTT/tt_embeddings.cpp:13-26,132)
 * output[tableidx[n]][rowidx[n]][:] += TT_row(indices[n]) for n < nnz; rows of `output`
 * that no index maps to are written as zeros (the reference returns at::zeros + RMW), so
 * `output` does not need to be initialised.  (tableidx, rowidx) may come in any order.
 * workspace: ttg_tt_workspace_bytes(shape, B, nnz) bytes, 256-byte aligned; the same
 * (shape, B, nnz) gives the same layout, which is what TTG_FLAG_PLAN_VALID relies on.
 * ----------------------------------------------------------------------------------  *
 * T = 4 tables whose T = 3 form (the first two cores contracted: p = (p0 p1, p2, p3), q = (q0 q1, q2, q3), ranks
 * (r2, r3)) has sorted / tensor-core kernels run on those; the contraction and its backward are part of the call,
 * and ttg_tt_workspace_bytes accounts for the merged core and its gradient.
 */
size_t ttg_tt_workspace_bytes(const ttg_shape* shape, int64_t B, int64_t nnz);

int ttg_tt_forward(const ttg_shape* shape, int64_t B, int64_t nnz,
                   const int64_t* indices, const int64_t* rowidx, const int64_t* tableidx,
                   const float* const* host_core_ptrs, /* host array of T device pointers */
                   float* output, void* workspace, size_t workspace_bytes, int32_t flags,
                   void* stream);

/* The index plan of a batch alone: sorted keys, output rows, group counters and bucket starts depend on
 * (indices, rowidx, tableidx) only, so a caller that knows the next batch -- the data loader's prefetch, which the
 * reference gets from DGL's DataLoader (sage_dgl_partition.py:141-154) -- builds its plan on another stream
 * while the current batch is still being processed, into the plan slot the current batch does not use
 * (TTG_FLAG_PLAN_SLOT1 selects the second slot), and then calls ttg_tt_forward with TTG_FLAG_PLAN_READY and
 * the same slot flag.  It replaces the index split at the head of the reference's forward
 * (FBTT/tt_embeddings_cuda.cu:757-921 / :1015-1027), which there runs inside every call.  Same workspace, same
 * (shape, B, nnz) as the forward that follows; TTG_ENOTSUP for shapes without the sorted kernels (the caller then
 * simply does not pass TTG_FLAG_PLAN_READY). */
int ttg_tt_plan(const ttg_shape* shape, int64_t B, int64_t nnz, const int64_t* indices,
                const int64_t* rowidx, const int64_t* tableidx, void* workspace, size_t workspace_bytes,
                int32_t flags, void* stream);

/* ------------------------------------------------------------------------------------
 * (b) backward + optimizer.
 * replaces: tt_embeddings_backward_cuda  FBTT/tt_embeddings_cuda.cu:421-654 behind the ops
 *           tt_dense_backward :656-686, tt_sgd_backward :688-719, tt_adagrad_backward
 *           :721-754 (FBTT/tt_embeddings.cpp:28-72,133-142)
 * d_cores[t] (fp32, same shape as core t) always receives the dense gradient (it is
 * overwritten, not accumulated).  optim == TTG_OPTIM_SGD additionally does
 * core -= lr * d_core; TTG_OPTIM_ADAGRAD does state += g*g; core -= lr*g/(sqrt(state)+eps)
 * over the WHOLE core (the reference's launch config skips tail rows, SURVEY 8a-6; we
 * implement the formula of FBTT/tt_embeddings_cuda.cu:381-419 on every row).
 * ---------------------------------------------------------------------------------- */
int ttg_tt_backward(const ttg_shape* shape, int32_t optim, float lr, float eps, int64_t B,
                    int64_t nnz, const int64_t* indices, const int64_t* rowidx,
                    const int64_t* tableidx, const float* d_output,
                    float* const* host_core_ptrs,      /* T device pointers, updated in place */
                    float* const* host_state_ptrs,     /* T device pointers or NULL          */
                    float* const* host_dcore_ptrs,     /* T device pointers (outputs)        */
                    void* workspace, size_t workspace_bytes, int32_t flags, void* stream);

/* (f-2) rows [first_row, first_row + num_rows) of a single-table TT matrix, in order: what the
 * reference obtains with forward(arange(N), arange(N + 1)) in its full-graph GCN / GAT steps and
 * in SAGE.inference (gcn_gat_partition.py:93-96, gnn_model.py:228-231).  No index arrays, no plan:
 * group table, then the forward row kernel on implicit keys; every staging buffer leaves as one
 * bulk copy.  Only for shapes with tensor-core kernels (TTG_ENOTSUP otherwise: the caller falls
 * back to ttg_tt_forward on an explicit index range). */
size_t ttg_tt_rows_range_workspace_bytes(const ttg_shape* shape);
int ttg_tt_rows_range(const ttg_shape* shape, int64_t first_row, int64_t num_rows,
                      const float* const* host_core_ptrs, float* output, void* workspace,
                      size_t workspace_bytes, int32_t flags, void* stream);

/* The optimizer step alone (what ttg_tt_backward fuses), for data-parallel training where the
 * dense gradients are all-reduced between the backward and the update.
 * replaces: update_tt_cores_sgd_kernel / update_tt_cores_adagrad_kernel
 *           FBTT/tt_embeddings_cuda.cu:381-419 (launches :612-651) */
int ttg_apply_optimizer(const ttg_shape* shape, int32_t optim, float lr, float eps,
                        float* const* host_core_ptrs, float* const* host_state_ptrs,
                        float* const* host_dcore_ptrs, void* stream);

/* Data-parallel exchange step over NVLink peer memory: the replacement of
 * DistributedDataParallel's all-reduce of the core gradients + the optimizer step
 * (sage_dgl_partition.py:235, FBTT/tt_embeddings_cuda.cu:381-419) by ONE kernel per step.
 *
 * Every rank (one process per GPU of one node) owns an exchange buffer of
 * ttg_peer_buffer_bytes(slot_floats) bytes: two gradient slots of slot_floats floats (each
 * rounded up to 256 bytes) followed by 64 flag words.  ttg_peer_alloc / _export on the owner,
 * ttg_peer_open on every other rank (the 64-byte handle travels by any host channel, e.g.
 * torch.distributed.all_gather_object); peer_buffers[r] is rank r's buffer as mapped HERE
 * (own allocation at r == rank).
 *
 * ttg_dp_exchange_update, called once per step on every rank after ttg_tt_backward(
 * TTG_OPTIM_DENSE) on the same stream: copies the dense gradients host_dcore_ptrs[t]
 * (seg_floats[t] floats each, a multiple of 4) into the slot of this step, signals the peers,
 * waits for all of them (bounded: after about 10 s the kernel gives up and records the step, see
 * ttg_peer_status), sums the `world` copies in rank order (bit-identical on all ranks), divides by
 * `world` and applies `optim` to the local cores (TTG_OPTIM_DENSE: only writes the mean to
 * mean_out, segments back to back; mean_out may also be given with the other modes).  The step
 * counter lives in the buffer: the call has no per-step argument and can be captured in a CUDA
 * graph.  Every rank must issue the same sequence of calls. */
size_t ttg_peer_buffer_bytes(int64_t slot_floats);
int ttg_peer_alloc(size_t bytes, void** ptr);
int ttg_peer_free(void* ptr);
int ttg_peer_export(void* ptr, void* handle64);
int ttg_peer_open(const void* handle64, void** ptr);
int ttg_peer_close(void* ptr);
int ttg_peer_status(const void* own_buffer, int64_t slot_floats, uint32_t* failed_epoch);
int ttg_dp_exchange_update(int32_t world, int32_t rank, void* const* peer_buffers, int32_t nseg,
                           const int64_t* seg_floats, const float* const* host_dcore_ptrs,
                           float* const* host_core_ptrs, float* const* host_state_ptrs,
                           int32_t optim, float lr, float eps, float* mean_out, void* stream);

/* ------------------------------------------------------------------------------------
 * (c) index path: LFU hash-table cache.
 * ---------------------------------------------------------------------------------- */
/* replaces: update_cache_state_cuda FBTT/tt_embeddings_cuda.cu:1083-1119 */
int ttg_update_cache_state(int64_t nnz, const int64_t* indices, int64_t hashtbl_size,
                           int64_t* hashtbl, int64_t* cache_freq, void* stream);

/* replaces: cache_populate_cuda FBTT/tt_embeddings_cuda.cu:1270-1347 (sort by frequency,
 * mark_popular_colidx_kernel :1122-1149, prefetch_cached_weights_cuda :1166-1268).
 * workspace: ttg_cache_populate_workspace_bytes(shape, hashtbl_size, cache_size). */
size_t ttg_cache_populate_workspace_bytes(const ttg_shape* shape, int64_t hashtbl_size,
                                          int64_t cache_size);
int ttg_cache_populate(const ttg_shape* shape, const float* const* host_core_ptrs,
                       int64_t hashtbl_size, int64_t* hashtbl, int64_t* cache_freq,
                       int32_t* cache_state, int64_t cache_size, float* cache_weight,
                       void* workspace, size_t workspace_bytes, void* stream);

/* replaces: preprocess_indices_sync_cuda FBTT/tt_embeddings_cuda.cu:1388-1507
 * (compute_rowidx_kernel :1349-1365, cache_lookup_kernel :1367-1386, 3x
 * cub::DevicePartition::Flagged :1448-1490).
 * Always writes rowidx/tableidx[nnz].  If warmup != 0 or num_tables != 1 nothing else is
 * written and *host_nnz_tt = nnz.  Otherwise part_colidx/part_rowidx/part_cache_loc[nnz]
 * receive [TT items in original order | cached items in REVERSED original order] and
 * *host_nnz_tt the number of TT items (stream is synchronised to produce it).
 * part_cache_loc entries of TT items are -1 (the reference leaves them uninitialised).
 * workspace: ttg_preprocess_workspace_bytes(nnz). */
size_t ttg_preprocess_workspace_bytes(int64_t nnz);
int ttg_preprocess_indices(int64_t nnz, int64_t num_offsets, const int64_t* colidx,
                           const int64_t* offsets, int32_t num_tables, int32_t warmup,
                           int64_t hashtbl_size, const int64_t* hashtbl,
                           const int32_t* cache_state, int64_t* rowidx, int64_t* tableidx,
                           int64_t* part_colidx, int64_t* part_rowidx,
                           int32_t* part_cache_loc, int32_t* host_nnz_tt, void* workspace,
                           size_t workspace_bytes, void* stream);

/* The cached / uncached split of preprocess_indices_sync_cuda (FBTT/tt_embeddings_cuda.cu:1388-1507: lookup
 * :1367-1386, partition :1440-1490) without the partition and without the host count it returns: tt_colidx[n] =
 * colidx[n] where the TT cores serve the entry, -1 (an id every TT kernel skips) where the cache does;
 * cache_loc[n] = the cache row or -1.  The TT ops then run on (tt_colidx, rowidx) and the cache ops on
 * (cache_loc, rowidx), both over all nnz entries: no stream synchronisation, so the module step can be
 * captured in a CUDA graph with the cache on.  The pybind-compatible op keeps its partition and its int. */
int ttg_cache_mark(int64_t nnz, const int64_t* colidx, int64_t hashtbl_size, const int64_t* hashtbl,
                   const int32_t* cache_state, int64_t* tt_colidx, int32_t* cache_loc, void* stream);

/* replaces: cache_forward_cuda FBTT/tt_embeddings_cuda.cu:1509-1583
 * output[rowidx[n]][:] += cache_weight[cache_locations[n]][:]  (accumulates; entries with a negative location
 * are skipped, here and in the cache backward ops) */
int ttg_cache_forward(int64_t nnz, int32_t D, const int32_t* cache_locations,
                      const int64_t* rowidx, const float* cache_weight, float* output,
                      void* stream);
/* replaces: cache_backward_sgd_cuda FBTT/tt_embeddings_cuda.cu:1585-1668 */
int ttg_cache_backward_sgd(int64_t nnz, int32_t D, const float* grad_output,
                           const int32_t* cache_locations, const int64_t* rowidx, float lr,
                           float* cache_weight, void* stream);
/* replaces: cache_backward_dense_cuda FBTT/tt_embeddings_cuda.cu:1670-1744
 * grad_cache_weight [cache_size][D] must be zero-initialised by the caller. */
int ttg_cache_backward_dense(int64_t nnz, int32_t D, const float* grad_output,
                             const int32_t* cache_locations, const int64_t* rowidx,
                             float* grad_cache_weight, void* stream);
/* replaces: cache_backward_rowwise_adagrad_approx_cuda FBTT/tt_embeddings_cuda.cu:1746-1846 */
int ttg_cache_backward_rowwise_adagrad_approx(int64_t nnz, int32_t D,
                                              const float* grad_output,
                                              const int32_t* cache_locations,
                                              const int64_t* rowidx, float lr, float eps,
                                              float* cache_optimizer_state,
                                              float* cache_weight, void* stream);

/* ------------------------------------------------------------------------------------
 * (c) Efficient_TT: prefix-reuse forward / dedup'd fused-SGD backward, 3 cores, one index
 * per output row, cores are 2-D [p[t]][cols_t].
 * replaces: Efficient_TT_forward_cuda Efficient_TT/efficient_tt_cuda.cu:243-377 and
 *           Fused_Extra_Efficient_TT_backward_sgd_cuda :1011-1247
 *           (Efficient_TT/efficient_kernel_wrap.cpp:16-28,63-80,83-89).
 * Index math is integer (the reference's float math is identical wherever it is exact,
 * SURVEY 8a-8).  No process-global scratch: the workspace is the caller's.
 * ---------------------------------------------------------------------------------- */
/* workspace for both Efficient_TT calls (index plan + dense gradient scratch) */
size_t ttg_eff_workspace_bytes(const ttg_shape* shape, int64_t batch);
int ttg_eff_forward(const ttg_shape* shape, int64_t batch, const int64_t* indices,
                    const float* const* host_core_ptrs, float* output, void* workspace,
                    size_t workspace_bytes, void* stream);
/* core_t[i_t] -= lr * (gradient slices summed over all rows); duplicates in `indices`
 * contribute once per occurrence, exactly like unique + inverse accumulation
 * (Efficient_TT/efficient_tt.py:132-133, efficient_tt_cuda.cu:970-987). */
int ttg_eff_backward_sgd(const ttg_shape* shape, int64_t batch, float lr,
                         const int64_t* indices, const float* d_output,
                         float* const* host_core_ptrs, void* workspace,
                         size_t workspace_bytes, int32_t flags, void* stream);

/* ------------------------------------------------------------------------------------
 * (d) neighbour aggregation on a sampled block (CSR by destination).
 * replaces: the SpMM inside dglnn.SAGEConv(..., 'mean') gnn_model.py:78-81,211-214 and
 *           dglnn.GraphConv(norm='both') gnn_model.py:287 (DGL 2.1.0, un-vendored).
 * out[v][:] = scale_v * sum_{e in [indptr[v], indptr[v+1])} w_e * x[indices[e]][:]
 *   mean != 0: scale_v = 1/deg(v) (0 rows stay 0);  mean == 0: scale_v = 1
 *   edge_weight may be NULL (w_e = 1).  F % 4 == 0 takes the 16-byte path, other widths
 *   (the 47-class output layer) a scalar one.
 * The backward is the same kernel on the transposed CSR (built once per block by the
 * caller) or ttg_spmm_csr_bwd which scatters with vector reductions.
 * ---------------------------------------------------------------------------------- */
int ttg_spmm_csr_fwd(int64_t num_dst, int32_t F, const int64_t* indptr,
                     const int32_t* indices, const float* edge_weight, int32_t mean,
                     const float* x, float* out, void* stream);
/* dx[indices[e]][:] += scale_v * w_e * dout[v][:]; dx [num_src][F] must be zeroed by caller */
int ttg_spmm_csr_bwd(int64_t num_dst, int32_t F, const int64_t* indptr,
                     const int32_t* indices, const float* edge_weight, int32_t mean,
                     const float* dout, float* dx, void* stream);

/* (d-2) mean over the in-neighbours of EVERY node of a whole graph (full-neighbour inference, the
 * layer-wise SAGE.inference of gnn_model.py:220-253), balanced by edges instead of by destinations:
 *   out[v][:] = (1 / deg(v)) * sum_{e in [indptr[v], indptr[v+1])} x[indices[e]][:]   (0 rows: deg 0)
 * Graph: indptr int64 [num_nodes + 1], indices int32 [num_edges] (ids < num_nodes); x, out fp32
 * [num_nodes][F], any F >= 1 (16-byte columns when F % 4 == 0).
 * ttg_mean_agg_plan cuts every row into work items of at most 256 edges (a per-node count, a scan, a
 * scatter); the plan depends on indptr alone and serves every later ttg_mean_agg on the same graph, at any
 * width.  Plan buffer: ttg_mean_agg_plan_bytes(num_nodes, num_edges) bytes, 16-byte aligned (bounded by
 * num_nodes + num_edges / 256 items of 16 bytes).  Workspace of either call:
 * ttg_mean_agg_workspace_bytes(num_nodes, num_edges, F) (plan build: any F >= 1); it holds the partial rows
 * of nodes with more than 256 in-edges, which a second pass sums in item order: no float atomics, the same
 * bits from every call.  Both queries return 0 for arguments out of range (num_nodes < 0 or >= 2^31,
 * num_edges < 0 or > 2^37, F <= 0).  The plan must come from the same indptr. */
size_t ttg_mean_agg_plan_bytes(int64_t num_nodes, int64_t num_edges);
size_t ttg_mean_agg_workspace_bytes(int64_t num_nodes, int64_t num_edges, int32_t F);
int ttg_mean_agg_plan(int64_t num_nodes, int64_t num_edges, const int64_t* indptr, void* plan,
                      size_t plan_bytes, void* workspace, size_t workspace_bytes, void* stream);
int ttg_mean_agg(int64_t num_nodes, int64_t num_edges, int32_t F, const int64_t* indptr,
                 const int32_t* indices, const void* plan, size_t plan_bytes, const float* x, float* out,
                 void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------
 * (f-4) the sparse part of GATConv on a CSR-by-destination block.
 * replaces: apply_edges(u_add_v) + leaky_relu + edge_softmax and update_all(u_mul_e, sum) of
 *           the reference's GATConv, gnn_model.py:413-420 (DGL 2.1, un-vendored: restated).
 * score / a / da / dscore fp32 [E][H] (edge-major), ft / dft fp32 [num_src][H*F],
 * out / dout fp32 [num_dst][H*F]; H <= 8.
 *   edge_softmax : a[e,h] = softmax over the in-edges of dst(e), per head
 *   head_spmm    : out[v,h,:] = sum_{e in N_in(v)} a[e,h] * ft[src(e),h,:]
 *   backward     : dscore = a * (da - sum_e a da);  dft += a * dout (dft zeroed by the caller),
 *                  da[e,h] = <dout[v,h,:], ft[src(e),h,:]>
 * ---------------------------------------------------------------------------------- */
int ttg_edge_softmax_csr_fwd(int64_t num_dst, int32_t H, const int64_t* indptr, const float* score,
                             float* out, void* stream);
int ttg_edge_softmax_csr_bwd(int64_t num_dst, int32_t H, const int64_t* indptr, const float* a,
                             const float* da, float* dscore, void* stream);
int ttg_head_spmm_csr_fwd(int64_t num_dst, int32_t H, int32_t F, const int64_t* indptr,
                          const int32_t* indices, const float* a, const float* ft, float* out,
                          void* stream);
int ttg_head_spmm_csr_bwd(int64_t num_dst, int32_t H, int32_t F, const int64_t* indptr,
                          const int32_t* indices, const float* a, const float* ft,
                          const float* dout, float* dft, float* da, void* stream);
/* the same backward without atomics, for callers that hold the block in source-major order as well (a static
 * graph transposes once): da as above, dft as a gather over (indptr_t [num_src + 1], dst_t [E], eid_t [E] = the
 * edge's position in the destination-major lists); every dft row is written, no zero fill needed */
int ttg_head_spmm_csr_bwd_gather(int64_t num_dst, int64_t num_src, int32_t H, int32_t F, const int64_t* indptr,
                                 const int32_t* indices, const float* a, const float* ft, const float* dout,
                                 const int64_t* indptr_t, const int32_t* dst_t, const int32_t* eid_t,
                                 float* dft, float* da, void* stream);

/* ------------------------------------------------------------------------------------
 * (f-1) neighbour sampling + block construction on the device, one GNN layer per call.
 * replaces: dgl.dataloading.NeighborSampler (uniform, without replacement) + to_block as the
 *           reference drives them, graphloader.py:245-261, sage_dgl_partition.py:141-154
 *           (DGL 2.1 is un-vendored: semantics restated, see csrc/sampler.cu).
 * Graph: CSR of in-neighbours, g_indptr int64 [num_nodes + 1], g_indices int32.
 * For every destination node (unique global ids, dst_nodes int64 [num_dst]) all its
 * in-neighbours are taken when there are at most `fanout`, else `fanout` distinct ones, the
 * draw being a pure function of (seed, node id).  Outputs (device):
 *   blk_indptr  int64 [num_dst + 1]              CSR by destination
 *   blk_indices int32 [capacity num_dst*fanout]  source ids local to the block
 *   src_nodes   int64 [capacity num_dst*(fanout+1)] global ids: the destination nodes first,
 *                                                then the new nodes in increasing id
 *   counts      int64 [2]                        {number of edges, number of source nodes}
 * No synchronisation: the caller reads `counts` when it needs the sizes on the host.
 * ---------------------------------------------------------------------------------- */
size_t ttg_sample_block_workspace_bytes(int64_t num_dst, int32_t fanout);
int ttg_sample_block(int64_t num_nodes, const int64_t* g_indptr, const int32_t* g_indices,
                     int64_t num_dst, const int64_t* dst_nodes, int32_t fanout, uint64_t seed,
                     int64_t* blk_indptr, int32_t* blk_indices, int64_t* src_nodes,
                     int64_t* counts, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------
 * (f-3) node reordering of a CSR graph (in-neighbour lists: indptr int64 [n + 1], indices int32).
 * replaces: dgl.reorder_graph(graph, 'custom' | 'rcmk' | 'metis', ...) as called at
 *           graphloader.py:370, 432, 440, 449 (DGL 2.1, un-vendored)
 *
 * ttg_permute_csr: the graph under the node permutation `perm` (new node i = old node perm[i],
 * DGL's nodes_perm convention); neighbour lists keep their order, ids are mapped through the
 * inverse permutation (also written to inverse_out when not NULL).  *bad_flag (device int32) is
 * set to 1 when perm holds an id outside [0, n); the outputs are then undefined.
 *
 * ttg_partition_grow: k parts grown from `seeds` by capacity-bounded label propagation over the
 * in-neighbour lists -- the stand-in for METIS-k (NOT the same partition; connected parts of at
 * most `cap` nodes).  Runs `sweeps` (even) synchronous sweeps; *changed (device int32) tells
 * whether any node joined a part in this call: call again with seeds == NULL (continue from
 * labels_a / sizes) until it stays 0.  labels_a holds the part of every node, -1 for nodes no
 * part could take.
 * ---------------------------------------------------------------------------------- */
size_t ttg_permute_csr_workspace_bytes(int64_t num_nodes);
int ttg_permute_csr(int64_t num_nodes, const int64_t* indptr, const int32_t* indices,
                    const int64_t* perm, int64_t* new_indptr, int32_t* new_indices,
                    int64_t* inverse_out, int32_t* bad_flag, void* workspace,
                    size_t workspace_bytes, void* stream);
int ttg_partition_grow(int64_t num_nodes, const int64_t* indptr, const int32_t* indices, int32_t k,
                       int32_t cap, const int64_t* seeds, int32_t sweeps, int32_t* labels_a,
                       int32_t* labels_b, int32_t* sizes, int32_t* changed, void* stream);

/* ttg_rcm_symmetrise + ttg_rcm_order: reverse Cuthill-McKee on the device, element for element the
 * permutation of scipy.sparse.csgraph.reverse_cuthill_mckee(adj, symmetric_mode=False) for adj = the CSR of
 * in-neighbour lists (DGL's 'rcmk').  The two calls split at the one host step, numpy.argsort of the degrees
 * (its tie order is numpy's):
 *
 *   ttg_rcm_symmetrise: scipy's adj + adj^T (num_edges = indptr[num_nodes]): sym_indptr int64 [n + 1],
 *     sym_indices int32 [max(2 * num_edges, 1)] (the first *sym_edges_out entries are written), degree int32 [n]
 *     (row length, + 1 for a self loop).  Rows are the distinct neighbours ascending when every in-list is
 *     strictly increasing, otherwise in reverse order of first appearance in [in-list, then every v whose
 *     in-list holds the row's node, increasing v].  *sym_edges_out is a HOST int64; the call synchronises the
 *     stream to read it.  TTG_EINVAL also when an id lies outside [0, n) or indptr exceeds num_edges.
 *   ttg_rcm_order: perm int64 [n] (perm[i] = old id of new node i) from the symmetrised lists, their degrees
 *     and rank_nodes int64 [n] = numpy.argsort(degree) (device copy).  stats_out (host int64 [2], may be NULL):
 *     {BFS levels, connected components}; phase_ms_out (host double [3], may be NULL): milliseconds spent on
 *     {components, BFS, final order}.  Synchronises the stream once per component round and per BFS level.
 *
 * Out of contract: 128 or more parallel edges between one pair of nodes (scipy's int8 sum wraps and drops the
 * entry) and in-lists of 2^31 or more entries.  Workspaces from the queries (0: sizes out of range). */
size_t ttg_rcm_symmetrise_workspace_bytes(int64_t num_nodes, int64_t num_edges);
int ttg_rcm_symmetrise(int64_t num_nodes, int64_t num_edges, const int64_t* indptr, const int32_t* indices,
                       int64_t* sym_indptr, int32_t* sym_indices, int32_t* degree, int64_t* sym_edges_out,
                       void* workspace, size_t workspace_bytes, void* stream);
size_t ttg_rcm_order_workspace_bytes(int64_t num_nodes);
int ttg_rcm_order(int64_t num_nodes, int64_t sym_edges, const int64_t* sym_indptr, const int32_t* sym_indices,
                  const int32_t* degree, const int64_t* rank_nodes, int64_t* perm, int64_t* stats_out,
                  double* phase_ms_out, void* workspace, size_t workspace_bytes, void* stream);

/* ttg_partition_kway: multilevel k-way partition (heavy-edge coarsening, grown initial parts, greedy
 * k-way refinement while uncoarsening) -- the role of METIS behind dgl.reorder_graph(g, 'metis',
 * permute_config={'k': k}) and dgl.metis_partition (graphloader.py:370, 377, 440).  HOST code like
 * METIS itself: every pointer is host memory, no stream.  The graph is symmetrised first (DGL does the
 * same), self loops and duplicate edges are allowed.  Every part holds at most
 * max(ceil(n / k), ubfactor * ceil(n / k)) nodes (ubfactor >= 1, METIS' ufactor; 1.03 is METIS'
 * default).  Deterministic in `seed`.  refine_passes <= 0 selects 10.  *edge_cut_out (may be NULL):
 * number of input edges whose two ends lie in different parts.  Not METIS' partition (csrc/kway_host.cu). */
int ttg_partition_kway(int64_t num_nodes, const int64_t* indptr, const int32_t* indices, int32_t k,
                       float ubfactor, uint64_t seed, int32_t refine_passes, int32_t* part_out,
                       int64_t* edge_cut_out);

/* ttg_partition_kway_initial: the host partitioner's initial step on a weighted graph (host memory, CSR with
 * edge weights adjw and vertex weights vw, both >= 1): eight grown partitions of the graph, each refined there with
 * the coarse-level bounds of a `total_nodes`-node graph (1.3 x the bounds above), the one with the smallest cut in
 * part_out [num_nodes].  The device partitioner below runs it on its coarsest level. */
int ttg_partition_kway_initial(int64_t num_nodes, const int64_t* xadj, const int32_t* adj, const int32_t* adjw,
                               const int32_t* vw, int64_t total_nodes, int32_t k, float ubfactor, uint64_t seed,
                               int32_t refine_passes, int32_t* part_out);

/* Multilevel k-way partition on the DEVICE (csrc/kway.cu): the scheme and the balance bounds of
 * ttg_partition_kway with every data-parallel step on the GPU, driven level by level by the caller
 * (reorder.kway_partition_device).  Not ttg_partition_kway's partition and not METIS'.  Deterministic in the seed.
 * Every call runs on `stream` in the caller's workspace (its *_workspace_bytes query), allocates nothing, and
 * refuses bad arguments before any CUDA call.  Weighted graphs are CSR: xadj int64 [n + 1], adj / adjw int32,
 * vw int32 [n].
 *   ttg_kway_symmetrise  the in-neighbour CSR (num_edges = indptr[num_nodes]) -> the undirected weighted graph
 *                        (weight = directed edges between the pair, no self loops, unit vertex weights); adj and
 *                        adjw hold 2 * num_edges entries, *sym_edges_out the used ones.  Ids out of range and an
 *                        indptr that is not a CSR of num_edges are refused (checked on the device).
 *   ttg_kway_coarsen     one level: matching (vertex weights <= maxvw; `level` varies the seed) and contraction.
 *                        cmap [n]; cxadj [n + 1], cadj / cadjw [num_edges], cvw [n] hold the coarse graph;
 *                        counts_out[0..1] = its vertex and edge counts (host memory; the call waits for them).
 *   ttg_kway_refine      part [n] on this level: first projected from coarse_part through cmap (both NULL: part
 *                        holds the labels already), then refined and rebalanced against the bounds of a
 *                        total_nodes-node graph (finest != 0: the exact bounds, which the call guarantees there;
 *                        else 1.3 x wider).  stats_out (host, may be NULL) [3]: label-propagation iterations,
 *                        local rebalancing rounds, exact fills.
 *   ttg_kway_edge_cut    *cut_out (host) = input edges whose ends lie in different parts. */
size_t ttg_kway_symmetrise_workspace_bytes(int64_t num_nodes, int64_t num_edges);
int ttg_kway_symmetrise(int64_t num_nodes, int64_t num_edges, const int64_t* indptr, const int32_t* indices,
                        int64_t* xadj, int32_t* adj, int32_t* adjw, int32_t* vw, int64_t* sym_edges_out,
                        void* workspace, size_t workspace_bytes, void* stream);
size_t ttg_kway_coarsen_workspace_bytes(int64_t num_nodes, int64_t num_edges);
int ttg_kway_coarsen(int64_t num_nodes, int64_t num_edges, const int64_t* xadj, const int32_t* adj,
                     const int32_t* adjw, const int32_t* vw, int32_t maxvw, uint64_t seed, int32_t level,
                     int32_t* cmap, int64_t* cxadj, int32_t* cadj, int32_t* cadjw, int32_t* cvw, int64_t* counts_out,
                     void* workspace, size_t workspace_bytes, void* stream);
size_t ttg_kway_refine_workspace_bytes(int64_t num_nodes, int32_t k);
int ttg_kway_refine(int64_t num_nodes, const int64_t* xadj, const int32_t* adj, const int32_t* adjw,
                    const int32_t* vw, int64_t total_nodes, int32_t k, float ubfactor, int32_t finest, uint64_t seed,
                    int32_t level, int32_t refine_passes, const int32_t* cmap, const int32_t* coarse_part,
                    int32_t* part, int64_t* stats_out, void* workspace, size_t workspace_bytes, void* stream);
size_t ttg_kway_edge_cut_workspace_bytes(void);
int ttg_kway_edge_cut(int64_t num_nodes, const int64_t* indptr, const int32_t* indices, const int32_t* part,
                      int64_t* cut_out, void* workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TTG_B200_H_ */
