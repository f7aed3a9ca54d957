"""Data-parallel plumbing for replicated TT cores (north star: "replicated cores and the
core-gradient allreduce over NCCL/NVLink").

The reference wraps the whole model in DistributedDataParallel (sage_dgl_partition.py:235), which
only all-reduces the cores when sparse=False; with the fused update (--sparse) its replicas would
silently diverge (SURVEY.md 3.5).  Here the exchange step is explicit and is the ONLY collective
on the path: one all-reduce (sum) over a flat fp32 buffer [d_core0 | d_core1 | d_core2 | extra],
divided by the world size, followed by the identical optimizer step on every rank
(ttg_apply_optimizer through the C ABI).  Works with the `nccl` backend on GPUs and with `gloo`
on CPU tensors (the latter is what the CPU tests exercise; the update itself needs CUDA).
"""
import ctypes as C
from typing import List, Optional, Sequence

import torch
import torch.distributed as dist

import _ttg


def shard_range(n: int, rank: int, world: int):
    """Contiguous, balanced split of n work units (seed nodes / rows) over `world` ranks: the
    first n % world ranks get one extra.  Same partitioning rule as DGL's use_ddp DataLoader
    without drop_last (sage_dgl_partition.py:144-154)."""
    base, extra = divmod(n, world)
    start = rank * base + min(rank, extra)
    return start, start + base + (1 if rank < extra else 0)


def epoch_permutation(n: int, epoch: int, seed: int = 0) -> torch.Tensor:
    """Same permutation on every rank for a given epoch (seeded), so the shards are disjoint."""
    g = torch.Generator()
    g.manual_seed(seed * 1000003 + epoch)
    return torch.randperm(n, generator=g)


def _shared_flat(tensors: Sequence[torch.Tensor]) -> Optional[torch.Tensor]:
    """The tensors as ONE flat view when they already sit back to back in one storage (what
    tt_dense_backward returns), else None."""
    if not tensors or any(not t.is_contiguous() for t in tensors):
        return None
    t0 = tensors[0]
    st = t0.untyped_storage().data_ptr()
    off = t0.storage_offset()
    for t in tensors:
        if t.dtype != t0.dtype or t.untyped_storage().data_ptr() != st or t.storage_offset() != off:
            return None
        off += t.numel()
    total = off - t0.storage_offset()
    return torch.as_strided(t0, (total,), (1,), t0.storage_offset())


def flatten(tensors: Sequence[torch.Tensor]) -> torch.Tensor:
    flat = _shared_flat(tensors)
    return flat if flat is not None else torch.cat([t.reshape(-1) for t in tensors])


def unflatten(flat: torch.Tensor, like: Sequence[torch.Tensor]) -> List[torch.Tensor]:
    out, off = [], 0
    for t in like:
        out.append(flat[off:off + t.numel()].view_as(t))
        off += t.numel()
    return out


def allreduce_mean(tensors: Sequence[torch.Tensor], group=None) -> List[torch.Tensor]:
    """One collective for all tensors; returns views into the reduced flat buffer."""
    flat = flatten(tensors)
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(flat, op=dist.ReduceOp.AVG if flat.is_cuda else dist.ReduceOp.SUM, group=group)
        if not flat.is_cuda:                       # gloo has no AVG
            flat.div_(dist.get_world_size(group))
    return unflatten(flat, tensors)


def apply_optimizer(tt_p_shapes, tt_q_shapes, tt_ranks, tt_cores: Sequence[torch.Tensor],
                    d_cores: Sequence[torch.Tensor], learning_rate: float, optimizer: str = "sgd",
                    eps: float = 1e-10, optimizer_state: Optional[Sequence[torch.Tensor]] = None):
    """core -= lr * g (sgd) or the Adagrad rule, in place, on torch's current stream."""
    cores = [c.data if isinstance(c, torch.nn.Parameter) else c for c in tt_cores]
    for i, (c, g) in enumerate(zip(cores, d_cores)):
        _ttg.require_cuda(c, "tt_cores[%d]" % i, torch.float32)
        _ttg.require_cuda(g, "d_cores[%d]" % i, torch.float32)
        if c.shape != g.shape:
            raise RuntimeError("apply_optimizer: gradient %d has the wrong shape" % i)
    num_tables = cores[0].size(0) if cores[0].dim() == 3 else 1
    shape = _ttg.make_shape(tt_p_shapes, tt_q_shapes, tt_ranks, num_tables)
    dev = cores[0].device
    optim = _ttg.OPTIM_SGD if optimizer == "sgd" else _ttg.OPTIM_ADAGRAD
    sp = None
    if optim == _ttg.OPTIM_ADAGRAD:
        sp = _ttg.ptr_array(optimizer_state)
    with _ttg.on_device(dev):
        cp, dp = _ttg.ptr_array(cores), _ttg.ptr_array(list(d_cores))
        rc = _ttg.lib().ttg_apply_optimizer(C.byref(shape), optim, float(learning_rate), float(eps),
                                            cp, sp, dp, _ttg.stream_of(dev))
        _ttg.check(rc, "apply_optimizer")
        _ttg.workspace.set_plan(dev, None)   # cores changed through raw pointers: the group table is stale


def map_peer_buffers(nbytes: int, device, group=None, what: str = "map_peer_buffers"):
    """One device buffer of `nbytes` per rank of `group`, every buffer mapped into every rank's address space
    (CUDA IPC through ttg_peer_alloc / _export / _open): (own buffer, the peer buffers opened here, a ctypes
    array of TTG_MAX_PEERS pointers with every rank's buffer as mapped here).  Collective, one process per GPU
    of one node.  A failure on ONE rank becomes a failure on ALL of them: all_gather_object carries each
    rank's error next to its handle, the open phase ends in an all-reduce(MIN) of an ok flag, and on
    disagreement every rank frees what it holds and raises RuntimeError."""
    import socket
    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    if world > _ttg.TTG_MAX_PEERS:
        raise RuntimeError("%s: at most %d ranks" % (what, _ttg.TTG_MAX_PEERS))
    lib = _ttg.lib()
    own_ptr, opened = None, []
    ptrs = (C.c_void_p * _ttg.TTG_MAX_PEERS)()
    err, handle = None, None
    with torch.cuda.device(device):
        own = C.c_void_p()
        if lib.ttg_peer_alloc(nbytes, C.byref(own)) != 0:
            err = "peer_alloc: " + _ttg.last_error()
        else:
            own_ptr = own.value
            h = (C.c_ubyte * _ttg.PEER_HANDLE_BYTES)()
            if lib.ttg_peer_export(own, h) != 0:
                err = "peer_export: " + _ttg.last_error()
            else:
                handle = bytes(h)
        mine = (socket.gethostname(), handle, err)
        everyone = [None] * world
        dist.all_gather_object(everyone, mine, group=group)
        errs = [e[2] for e in everyone if e[2]]
        if not errs and any(e[0] != mine[0] for e in everyone):
            errs = ["the ranks are not on one node"]
        if errs:
            release_peer_buffers(own_ptr, opened)
            raise RuntimeError("%s: %s" % (what, errs[0]))
        ok = 1
        for r, (_, h, _) in enumerate(everyone):
            if r == rank:
                ptrs[r] = own_ptr
                continue
            p = C.c_void_p()
            buf = (C.c_ubyte * _ttg.PEER_HANDLE_BYTES).from_buffer_copy(h)
            if lib.ttg_peer_open(buf, C.byref(p)) != 0:
                ok, err = 0, "peer_open(rank %d): %s" % (r, _ttg.last_error())
                break
            ptrs[r] = p.value
            opened.append(p.value)
        flag = torch.tensor([ok], dtype=torch.int32, device=device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)   # also: every buffer is mapped everywhere
        if int(flag.item()) == 0:
            release_peer_buffers(own_ptr, opened)
            raise RuntimeError("%s: %s" % (what, err or "a peer could not map the buffers"))
    return own_ptr, opened, ptrs


def release_peer_buffers(own, opened) -> None:
    """Undo map_peer_buffers on this rank: close the peer mappings, free the own buffer."""
    lib = _ttg.lib()
    for p in opened:
        lib.ttg_peer_close(C.c_void_p(p))
    if own is not None:
        lib.ttg_peer_free(C.c_void_p(own))


class PeerExchange:
    """The exchange step without NCCL: gradient slots that every GPU of the node has mapped, and
    one kernel per step that publishes this rank's gradients, waits for the peers, sums the copies
    in rank order and applies the optimizer (ttg_dp_exchange_update, csrc/peer.cu).  One object
    per replicated TT table.

        xchg = PeerExchange(module.tt_cores)          # collective: every rank of `group`
        ... loss.backward()                           # dense gradients, anywhere
        xchg.step(grads, module.tt_cores, "sgd", lr)  # every rank, same sequence of calls

    step() has no per-step host state (the step counter lives on the device), so it can be
    captured in a CUDA graph together with the forward and backward.  Raises RuntimeError when
    the ranks are not GPUs of one node with peer access."""

    def __init__(self, tt_cores: Sequence[torch.Tensor], group=None):
        if not (dist.is_available() and dist.is_initialized()):
            raise RuntimeError("PeerExchange: torch.distributed is not initialised")
        cores = [c.data if isinstance(c, torch.nn.Parameter) else c for c in tt_cores]
        for i, c in enumerate(cores):
            _ttg.require_cuda(c, "tt_cores[%d]" % i, torch.float32)
            if c.numel() % 4:
                raise RuntimeError("PeerExchange: core %d has %d elements, not a multiple of 4"
                                   % (i, c.numel()))
        self.group = group
        self.world = dist.get_world_size(group)
        self.rank = dist.get_rank(group)
        self.device = cores[0].device
        self.sizes = [c.numel() for c in cores]
        self.total = sum(self.sizes)
        self.seg = (C.c_int64 * len(self.sizes))(*self.sizes)
        self.nbytes = _ttg.lib().ttg_peer_buffer_bytes(self.total)
        self.own, self.opened, self.ptrs = map_peer_buffers(self.nbytes, self.device, group, "PeerExchange")

    def _release(self) -> None:
        release_peer_buffers(self.own, self.opened)
        self.own, self.opened = None, []

    def step(self, d_cores: Sequence[torch.Tensor], tt_cores: Sequence[torch.Tensor],
             optimizer: str = "sgd", learning_rate: float = 0.0, eps: float = 1e-10,
             optimizer_state: Optional[Sequence[torch.Tensor]] = None,
             mean_out: Optional[torch.Tensor] = None) -> Optional[torch.Tensor]:
        """optimizer: "sgd" | "adagrad" | "dense" (only the mean gradient, returned as a flat
        tensor).  Every rank must call step() the same number of times."""
        optim = {"sgd": _ttg.OPTIM_SGD, "adagrad": _ttg.OPTIM_ADAGRAD, "dense": _ttg.OPTIM_DENSE}[optimizer]
        cores = [c.data if isinstance(c, torch.nn.Parameter) else c for c in tt_cores]
        grads = []
        for i, (g, n) in enumerate(zip(d_cores, self.sizes)):
            g = _ttg.require_cuda(g.detach(), "d_cores[%d]" % i, torch.float32)
            if g.numel() != n:
                raise RuntimeError("PeerExchange.step: gradient %d has the wrong size" % i)
            grads.append(g)
        if optim == _ttg.OPTIM_DENSE and mean_out is None:
            mean_out = torch.empty(self.total, dtype=torch.float32, device=self.device)
        sp = _ttg.ptr_array(optimizer_state) if optim == _ttg.OPTIM_ADAGRAD else None
        with _ttg.on_device(self.device):
            rc = _ttg.lib().ttg_dp_exchange_update(
                self.world, self.rank, self.ptrs, len(self.sizes), self.seg, _ttg.ptr_array(grads),
                _ttg.ptr_array(cores), sp, optim, float(learning_rate), float(eps),
                _ttg.ptr(mean_out), _ttg.stream_of(self.device))
            _ttg.check(rc, "dp_exchange_update")
            if optim != _ttg.OPTIM_DENSE:
                _ttg.workspace.set_plan(self.device, None)   # cores changed: the group table is stale
        return mean_out

    def failed_epoch(self) -> int:
        """0, or the step at which a peer did not arrive within the kernel's wait budget
        (synchronises the device)."""
        v = C.c_uint32(0)
        torch.cuda.synchronize(self.device)
        _ttg.check(_ttg.lib().ttg_peer_status(C.c_void_p(self.own), self.total, C.byref(v)), "peer_status")
        return int(v.value)

    def close(self) -> None:
        if self.own is None:
            return
        torch.cuda.synchronize(self.device)
        dist.barrier(group=self.group)               # nobody still reads what is about to go away
        self._release()


def dp_backward_step(module, d_cores: Sequence[torch.Tensor], group=None,
                     exchange: Optional[PeerExchange] = None):
    """All-reduce the dense core gradients of a TTEmbeddingBag and apply its own optimizer:
    the data-parallel equivalent of the fused --sparse update.  With `exchange` the whole step is
    one kernel over NVLink peer memory, otherwise one NCCL all-reduce plus the update."""
    from FBTT.tt_embeddings_ops import OptimType
    sgd = module.optimizer in (OptimType.SGD, OptimType.EXACT_SGD)
    if exchange is not None:
        exchange.step(d_cores, list(module.tt_cores), "sgd" if sgd else "adagrad",
                      module.learning_rate, module.eps, None if sgd else list(module.optimizer_state))
        return None
    reduced = allreduce_mean(d_cores, group)
    apply_optimizer(module.tt_p_shapes, module.tt_q_shapes, module.tt_ranks, list(module.tt_cores),
                    reduced, module.learning_rate, "sgd" if sgd else "adagrad", module.eps,
                    None if sgd else list(module.optimizer_state))
    return reduced


def merged_key_counts(keys: torch.Tensor, counts: torch.Tensor, group=None):
    """Union of every rank's (key, count) pairs with the counts of equal keys added: the access statistics of the
    whole job instead of one rank's shard of the seeds.  Collective; every rank returns the same sorted keys and
    their summed counts.  (The reference populates each replica's cache from its own counts,
    FBTT/tt_embeddings_ops.py:816-830 under sage_dgl_partition.py:359-361, so the replicas cache different
    rows; SURVEY 8e.)"""
    keys = keys.reshape(-1).to(torch.int64)
    counts = counts.reshape(-1).to(torch.int64)
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        world = dist.get_world_size(group)
        n = torch.tensor([keys.numel()], dtype=torch.int64, device=keys.device)
        sizes = [torch.zeros_like(n) for _ in range(world)]
        dist.all_gather(sizes, n, group=group)
        cap = max(int(x.item()) for x in sizes)
        pad_k = torch.full((cap,), -1, dtype=torch.int64, device=keys.device)
        pad_c = torch.zeros((cap,), dtype=torch.int64, device=keys.device)
        pad_k[:keys.numel()] = keys
        pad_c[:keys.numel()] = counts
        all_k = [torch.empty_like(pad_k) for _ in range(world)]
        all_c = [torch.empty_like(pad_c) for _ in range(world)]
        dist.all_gather(all_k, pad_k, group=group)
        dist.all_gather(all_c, pad_c, group=group)
        keys = torch.cat([k[:int(m.item())] for k, m in zip(all_k, sizes)])
        counts = torch.cat([c[:int(m.item())] for c, m in zip(all_c, sizes)])
    uk, inv = torch.unique(keys, return_inverse=True)
    uc = torch.zeros(uk.numel(), dtype=torch.int64, device=keys.device).index_add_(0, inv, counts)
    return uk, uc


def merge_lfu_statistics(module, group=None) -> int:
    """Replace the LFU table of a cached TTEmbeddingBag (hashtbl, cache_freq) by the merged statistics of all
    ranks, so that the cache_populate() that follows picks the same rows on every replica.  Call it on every
    rank right before module.cache_populate().  Returns the number of distinct keys."""
    import tt_embeddings
    if not getattr(module, "use_cache", False):
        return 0
    tbl, freq = module.hashtbl, module.cache_freq
    used = tbl >= 0
    uk, uc = merged_key_counts(tbl[used], freq[used], group)
    if uk.numel() > tbl.numel():
        # more distinct rows than slots: keep the most frequent ones (ties by key, the same on every rank)
        order = torch.argsort(uc * (int(uk.max().item()) + 1) - uk, descending=True)[:tbl.numel()]
        order, _ = torch.sort(order)
        uk, uc = uk[order], uc[order]
    tbl.fill_(-1)
    freq.fill_(0)
    tt_embeddings.update_cache_state(uk, tbl, freq)        # every key once
    slots = (tbl >= 0).nonzero(as_tuple=True)[0]
    pos = torch.searchsorted(uk, tbl[slots])
    freq[slots] = uc[pos].to(freq.dtype)
    return int(uk.numel())
