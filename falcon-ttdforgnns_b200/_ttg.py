"""ctypes binding of libttg_b200.so (include/ttg_b200.h) + the small amount of host logic the
ops share: shape structs, the per-device workspace, error translation.

PyTorch is used for device memory and streams only; every computation is a call through the
C ABI.  There is no CPU or eager fallback: if the library is missing, lib() raises.
"""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libttg_b200.so")
_lib = None

TTG_MAX_CORES = 4
TTG_MAX_PEERS = 8
PEER_HANDLE_BYTES = 64
OPTIM_SGD, OPTIM_ADAGRAD, OPTIM_DENSE = 0, 1, 2
FLAG_FORCE_GENERIC, FLAG_PLAN_VALID, FLAG_DETERMINISTIC, FLAG_TF32, FLAG_FFMA = 1, 2, 4, 8, 16
FLAG_MMA_SYNC, FLAG_TCGEN05, FLAG_PLAN_READY, FLAG_PLAN_SLOT1, FLAG_SHARE_SMS = 32, 64, 128, 256, 512
FLAG_RIGHT = 1024


class Shape(C.Structure):
    _fields_ = [("T", C.c_int32), ("num_tables", C.c_int32), ("p", C.c_int32 * TTG_MAX_CORES),
                ("q", C.c_int32 * TTG_MAX_CORES), ("r", C.c_int32 * (TTG_MAX_CORES + 1))]


_vp, _i64, _i32, _f32, _sz = C.c_void_p, C.c_int64, C.c_int32, C.c_float, C.c_size_t
_SP = C.POINTER(Shape)

# name -> (restype, argtypes); exactly the entry points include/ttg_b200.h declares
SIGNATURES = {
    "ttg_last_error": (C.c_char_p, []),
    "ttg_version": (C.c_int, []),
    "ttg_launch_count": (_i64, []),
    "ttg_profile_enable": (C.c_int, [_i32]),
    "ttg_profile_read": (C.c_int, [_i32, C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    "ttg_profile_name": (C.c_char_p, [_i32]),
    "ttg_apply_optimizer": (C.c_int, [_SP, _i32, _f32, _f32, _vp, _vp, _vp, _vp]),
    "ttg_peer_buffer_bytes": (_sz, [_i64]),
    "ttg_peer_alloc": (C.c_int, [_sz, C.POINTER(C.c_void_p)]),
    "ttg_peer_free": (C.c_int, [_vp]),
    "ttg_peer_export": (C.c_int, [_vp, _vp]),
    "ttg_peer_open": (C.c_int, [_vp, C.POINTER(C.c_void_p)]),
    "ttg_peer_close": (C.c_int, [_vp]),
    "ttg_peer_status": (C.c_int, [_vp, _i64, C.POINTER(C.c_uint32)]),
    "ttg_dp_exchange_update": (C.c_int, [_i32, _i32, _vp, _i32, C.POINTER(C.c_int64), _vp, _vp, _vp,
                                         _i32, _f32, _f32, _vp, _vp]),
    "ttg_tt_workspace_bytes": (_sz, [_SP, _i64, _i64]),
    "ttg_tt_forward": (C.c_int, [_SP, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _i32, _vp]),
    "ttg_tt_plan": (C.c_int, [_SP, _i64, _i64, _vp, _vp, _vp, _vp, _sz, _i32, _vp]),
    "ttg_tt_backward": (C.c_int, [_SP, _i32, _f32, _f32, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp,
                                  _vp, _vp, _sz, _i32, _vp]),
    "ttg_tt_rows_range_workspace_bytes": (_sz, [_SP]),
    "ttg_tt_rows_range": (C.c_int, [_SP, _i64, _i64, _vp, _vp, _vp, _sz, _i32, _vp]),
    "ttg_update_cache_state": (C.c_int, [_i64, _vp, _i64, _vp, _vp, _vp]),
    "ttg_cache_populate_workspace_bytes": (_sz, [_SP, _i64, _i64]),
    "ttg_cache_populate": (C.c_int, [_SP, _vp, _i64, _vp, _vp, _vp, _i64, _vp, _vp, _sz, _vp]),
    "ttg_preprocess_workspace_bytes": (_sz, [_i64]),
    "ttg_preprocess_indices": (C.c_int, [_i64, _i64, _vp, _vp, _i32, _i32, _i64, _vp, _vp, _vp, _vp,
                                         _vp, _vp, _vp, C.POINTER(C.c_int32), _vp, _sz, _vp]),
    "ttg_cache_mark": (C.c_int, [_i64, _vp, _i64, _vp, _vp, _vp, _vp, _vp]),
    "ttg_cache_forward": (C.c_int, [_i64, _i32, _vp, _vp, _vp, _vp, _vp]),
    "ttg_cache_backward_sgd": (C.c_int, [_i64, _i32, _vp, _vp, _vp, _f32, _vp, _vp]),
    "ttg_cache_backward_dense": (C.c_int, [_i64, _i32, _vp, _vp, _vp, _vp, _vp]),
    "ttg_cache_backward_rowwise_adagrad_approx": (C.c_int, [_i64, _i32, _vp, _vp, _vp, _f32, _f32,
                                                            _vp, _vp, _vp]),
    "ttg_eff_workspace_bytes": (_sz, [_SP, _i64]),
    "ttg_eff_forward": (C.c_int, [_SP, _i64, _vp, _vp, _vp, _vp, _sz, _vp]),
    "ttg_eff_backward_sgd": (C.c_int, [_SP, _i64, _f32, _vp, _vp, _vp, _vp, _sz, _i32, _vp]),
    "ttg_spmm_csr_fwd": (C.c_int, [_i64, _i32, _vp, _vp, _vp, _i32, _vp, _vp, _vp]),
    "ttg_spmm_csr_bwd": (C.c_int, [_i64, _i32, _vp, _vp, _vp, _i32, _vp, _vp, _vp]),
    "ttg_mean_agg_plan_bytes": (_sz, [_i64, _i64]),
    "ttg_mean_agg_workspace_bytes": (_sz, [_i64, _i64, _i32]),
    "ttg_mean_agg_plan": (C.c_int, [_i64, _i64, _vp, _vp, _sz, _vp, _sz, _vp]),
    "ttg_mean_agg": (C.c_int, [_i64, _i64, _i32, _vp, _vp, _vp, _sz, _vp, _vp, _vp, _sz, _vp]),
    "ttg_edge_softmax_csr_fwd": (C.c_int, [_i64, _i32, _vp, _vp, _vp, _vp]),
    "ttg_edge_softmax_csr_bwd": (C.c_int, [_i64, _i32, _vp, _vp, _vp, _vp, _vp]),
    "ttg_head_spmm_csr_fwd": (C.c_int, [_i64, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "ttg_head_spmm_csr_bwd": (C.c_int, [_i64, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "ttg_head_spmm_csr_bwd_gather": (C.c_int, [_i64, _i64, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                               _vp, _vp]),
    "ttg_permute_csr_workspace_bytes": (_sz, [_i64]),
    "ttg_permute_csr": (C.c_int, [_i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "ttg_rcm_symmetrise_workspace_bytes": (_sz, [_i64, _i64]),
    "ttg_rcm_symmetrise": (C.c_int, [_i64, _i64, _vp, _vp, _vp, _vp, _vp, C.POINTER(C.c_int64), _vp, _sz, _vp]),
    "ttg_rcm_order_workspace_bytes": (_sz, [_i64]),
    "ttg_rcm_order": (C.c_int, [_i64, _i64, _vp, _vp, _vp, _vp, _vp, C.POINTER(C.c_int64), C.POINTER(C.c_double),
                                _vp, _sz, _vp]),
    "ttg_partition_grow": (C.c_int, [_i64, _vp, _vp, _i32, _i32, _vp, _i32, _vp, _vp, _vp, _vp, _vp]),
    "ttg_partition_kway": (C.c_int, [_i64, _vp, _vp, _i32, _f32, C.c_uint64, _i32, _vp, C.POINTER(C.c_int64)]),
    "ttg_partition_kway_initial": (C.c_int, [_i64, _vp, _vp, _vp, _vp, _i64, _i32, _f32, C.c_uint64, _i32, _vp]),
    "ttg_kway_symmetrise_workspace_bytes": (_sz, [_i64, _i64]),
    "ttg_kway_symmetrise": (C.c_int, [_i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, C.POINTER(C.c_int64), _vp, _sz, _vp]),
    "ttg_kway_coarsen_workspace_bytes": (_sz, [_i64, _i64]),
    "ttg_kway_coarsen": (C.c_int, [_i64, _i64, _vp, _vp, _vp, _vp, _i32, C.c_uint64, _i32, _vp, _vp, _vp, _vp, _vp,
                                   C.POINTER(C.c_int64), _vp, _sz, _vp]),
    "ttg_kway_refine_workspace_bytes": (_sz, [_i64, _i32]),
    "ttg_kway_refine": (C.c_int, [_i64, _vp, _vp, _vp, _vp, _i64, _i32, _f32, _i32, C.c_uint64, _i32, _i32, _vp, _vp,
                                  _vp, C.POINTER(C.c_int64), _vp, _sz, _vp]),
    "ttg_kway_edge_cut_workspace_bytes": (_sz, []),
    "ttg_kway_edge_cut": (C.c_int, [_i64, _vp, _vp, _vp, C.POINTER(C.c_int64), _vp, _sz, _vp]),
    "ttg_sample_block_workspace_bytes": (_sz, [_i64, _i32]),
    "ttg_sample_block": (C.c_int, [_i64, _vp, _vp, _i64, _vp, _i32, C.c_uint64, _vp, _vp, _vp, _vp,
                                   _vp, _sz, _vp]),
}


def lib():
    """Load the CUDA library; fail loudly if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "ttg_b200: %s is missing -- build it with `python falcon-ttdforgnns_b200/build.py` "
                "(there is no CPU fallback)" % LIB_PATH)
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def last_error():
    msg = lib().ttg_last_error()
    return msg.decode() if msg else "?"


def check(rc, what):
    if rc != 0:
        msg = lib().ttg_last_error()
        raise RuntimeError("%s failed (code %d): %s" % (what, rc, msg.decode() if msg else "?"))


_shape_cache = {}


def make_shape(tt_p_shapes, tt_q_shapes, tt_ranks, num_tables=1):
    """ttg_shape struct for (p, q, ranks, num_tables); built once per distinct table."""
    key = (tuple(tt_p_shapes), tuple(tt_q_shapes), tuple(tt_ranks), int(num_tables))
    s = _shape_cache.get(key)
    if s is not None:
        return s
    T = len(tt_p_shapes)
    ranks = [int(x) for x in tt_ranks]
    if len(ranks) == T - 1:
        ranks = [1] + ranks + [1]
    if not (2 <= T <= TTG_MAX_CORES and len(tt_q_shapes) == T and len(ranks) == T + 1):
        raise RuntimeError("ttg_b200: need 2..4 cores with len(p) == len(q) == len(ranks) - 1")
    s = Shape()
    s.T = T
    s.num_tables = int(num_tables)
    for t in range(T):
        s.p[t] = int(tt_p_shapes[t])
        s.q[t] = int(tt_q_shapes[t])
    for t in range(T + 1):
        s.r[t] = ranks[t]
    s.key = key          # python-side identity of the table shape (plan keys, size caches)
    if len(_shape_cache) < 256:
        _shape_cache[key] = s
    return s


_ws_bytes_cache = {}


def tt_workspace_bytes(shape, B, nnz):
    """ttg_tt_workspace_bytes, memoised (the size is a pure function of its arguments)."""
    key = (getattr(shape, "key", None), int(B), int(nnz))
    n = _ws_bytes_cache.get(key) if key[0] is not None else None
    if n is None:
        n = lib().ttg_tt_workspace_bytes(C.byref(shape), B, nnz)
        if key[0] is not None and len(_ws_bytes_cache) < 4096:
            _ws_bytes_cache[key] = n
    return n


class on_device:
    """`with torch.cuda.device(dev)` that does nothing when dev is already current (the usual
    case: one process per GPU); switching devices through torch costs ~10 us per call."""

    def __init__(self, dev):
        idx = dev.index
        self.ctx = None if (idx is None or idx == torch.cuda.current_device()) else torch.cuda.device(dev)

    def __enter__(self):
        if self.ctx is not None:
            self.ctx.__enter__()

    def __exit__(self, *a):
        if self.ctx is not None:
            self.ctx.__exit__(*a)
        return False


def ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def ptr_array(tensors):
    """Host array of device pointers (kept alive by the caller holding the return value)."""
    arr = (C.c_void_p * TTG_MAX_CORES)()
    for i, t in enumerate(tensors):
        arr[i] = t.data_ptr()
    return arr


def stream_of(device):
    """torch's current stream on `device` as a raw cudaStream_t (the private getter skips the
    Stream object construction, which costs more than a kernel launch)."""
    idx = device.index if device.index is not None else torch.cuda.current_device()
    try:
        return C.c_void_p(torch._C._cuda_getCurrentRawStream(idx))
    except AttributeError:  # older / newer torch without the private getter
        return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def require_cuda(t, name, dtype=None):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError("ttg_b200: %s must be a CUDA tensor (no CPU path exists)" % name)
    if dtype is not None and t.dtype != dtype:
        raise RuntimeError("ttg_b200: %s must have dtype %s, got %s" % (name, dtype, t.dtype))
    if not t.is_contiguous():
        raise RuntimeError("ttg_b200: %s must be contiguous" % name)
    return t


class _Workspace:
    """One growable scratch buffer per device.  `plan_key` remembers which (indices, shape)
    the sorted plan inside currently belongs to, so a backward that follows its forward skips
    the sort (TTG_FLAG_PLAN_VALID)."""

    def __init__(self):
        self.buf = {}
        self.plan_key = {}
        self.keep = {}   # tensors the plan was built from: kept alive so their addresses
                         # cannot be recycled while the key is still trusted
        self.ready = {}  # (device, slot) -> (key, keep): index plans ttg_tt_plan built ahead of their forward
        self.layout = {} # device -> (shape, B, nnz) the buffer is currently carved for: the C side lays the
                         # workspace out as a function of these, so a plan prepared under one layout must
                         # neither be used nor be BUILT (it runs beside the current batch) under another

    def get(self, device, nbytes):
        key = (device.type, device.index)
        b = self.buf.get(key)
        if b is None or b.numel() < nbytes:
            b = torch.empty(int(nbytes * 1.25) + 1024, dtype=torch.uint8, device=device)
            self.buf[key] = b
            self.plan_key[key] = None
            for k in [k for k in self.ready if k[:2] == key]:   # plans lived in the old buffer
                del self.ready[k]
        return b

    def plan(self, device):
        return self.plan_key.get((device.type, device.index))

    def same_layout(self, device, layout, adopt=True):
        """Is the buffer carved for `layout`?  adopt: make it so (dropping the plans prepared under the old one)."""
        key = (device.type, device.index)
        cur = self.layout.get(key)
        if cur == layout:
            return True
        if adopt:
            self.layout[key] = layout
            for k in [k for k in self.ready if k[:2] == key]:
                del self.ready[k]
            self.plan_key[key] = None
        return cur is None

    def set_ready(self, device, slot, key, keep=None):
        self.ready[(device.type, device.index, int(slot))] = (key, keep)

    def ready_slot(self, device, key):
        """Plan slot that holds the ready plan `key`, or None."""
        for slot in (0, 1):
            e = self.ready.get((device.type, device.index, slot))
            if e is not None and e[0] == key:
                return slot
        return None

    def drop_ready(self, device, slot):
        self.ready.pop((device.type, device.index, int(slot)), None)

    def set_plan(self, device, key, keep=None):
        self.plan_key[(device.type, device.index)] = key
        self.keep[(device.type, device.index)] = keep


workspace = _Workspace()


def index_key_of(tag, indices, rowidx, nnz, B, shape_tuple):
    """Identity of an index plan alone (no stream: it is handed from the stream that built it to the one that
    uses it through an event the caller owns; no cores: the plan does not depend on them)."""
    return (tag, indices.data_ptr(), indices._version, rowidx.data_ptr(), rowidx._version, int(nnz), int(B),
            shape_tuple)


def plan_key_of(tag, indices, rowidx, nnz, B, shape_tuple, cores=()):
    """Identity of an index plan + group table: the stream it was built on, the index tensors (address and
    version counter), the sizes, the table shape and the cores the group table was computed from.  Pass the
    cores as the caller holds them (nn.Parameter or its .detach()): `.data` makes a tensor with its own
    version counter that never moves.  Updates through raw pointers (ttg_apply_optimizer, the peer exchange)
    do not bump any counter: dp.apply_optimizer / PeerExchange.step clear the plan themselves."""
    dev = indices.device
    try:
        stream = int(torch._C._cuda_getCurrentRawStream(dev.index if dev.index is not None
                                                        else torch.cuda.current_device()))
    except AttributeError:
        stream = int(torch.cuda.current_stream(dev).cuda_stream)
    return (tag, stream, indices.data_ptr(), indices._version, rowidx.data_ptr(), rowidx._version,
            int(nnz), int(B), shape_tuple,
            tuple((c.data_ptr(), c._version) for c in cores))
